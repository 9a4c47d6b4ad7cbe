#!/usr/bin/env python
"""bench.py -- one-shot localization throughput (BASELINE.json metric: queries/s vs DB size,
vote-kernel HBM GB/s).

A "step" is one pass of the hot path over one batch of synthetic queries:
  descriptor construction for every query scan (stage 2) + vote / top-k / match lists /
  geometric verification against the keyframe database (stages 3-4), i.e.
  BuildSingleScanSTD + SearchLoop per query (R/src/semantic_graph_localization.cpp:590-602).

Workload of the headline line (config.workload): BASELINE.json configs[3] -- 100k-keyframe
synthetic city DB, 1,024-query batch.  It fits one B200, so N=1 runs it unsharded; N>1 shards
the DB by keyframe range (strong scaling: total work is fixed), merges per-shard top-k lists
with ncclAllGather and gathers verified candidates back.

  value      queries/s, query nodes already resident in HBM
  e2e        queries/s through the C ABI with HOST buffers (H2D of the node arrays + D2H of
             loop results and candidates inside the timed region)
  roofline   the vote kernel against HBM.  `achieved` = one-pass byte bound / CUDA-event
             time of the kernel, bound = 16 B x entries of the DISTINCT buckets the batch probes
             (each read once) + 32 B x query descriptors + 16 B x probes (bucket headers) +
             4 B x nq x F (vote rows written once); `traffic` = ncu DRAM bytes of one launch from
             profiles/r02_traffic.json (keyed by kernel / workload / source hash);
             `reread_factor` = traffic / bound.  The SURVEY 8d per-probe model is reported
             beside it (`per_probe_model_*`): it is what the streaming kernel moves, not a
             bound for the join.
  db_sweep   the "vs DB size" half of the metric: 1k / 10k / 100k keyframes (N=1 only)
  stage1     instance extraction (voxel hashing) on a batch of labelled scans: scans/s and
             GB/s on 24 B/point (N=1 only)
  parity_checked  one warm-up step is run with the exact FP64 streaming kernel and must give
             byte-identical vote rows and candidates
  cpu_baseline    the oracle (CPU port of the reference) on a bounded sample, plus the
             REFERENCE BUILD (oracle/_ref: the reference's own STDesc.cpp compiled in place) at 4 / 8
             threads on the 1k-keyframe DB

--impl reference times the CPU implementation on the SAME 100k-keyframe database: the oracle
port (the reference's own code cannot hold it: `double match_array[MAX_FRAME_N=20000]`,
R/src/STDesc.cpp:323, and ~0.5 KB per STDesc); each step is a bounded number of queries.
"""
import argparse
import ctypes
import hashlib
import json
import os
import subprocess
import sys
import threading
import time
import zlib

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOAD = "configs[3]: 100k-keyframe synthetic city DB, 1024-query batch"
METRIC = "one-shot localization queries/s"
STAT_KEYS = ("Q", "P", "Pfound", "E", "M")


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--keyframes", type=int, default=100000)
    ap.add_argument("--queries", type=int, default=1024)
    ap.add_argument("--cpu-keyframes", type=int, default=8192, help="DB prefix used by the cpu_baseline sample of our arm")
    ap.add_argument("--cpu-queries", type=int, default=8)
    ap.add_argument("--ref-budget-s", type=float, default=150.0, help="--impl reference: target for the timed + warm-up steps")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip db_sweep / stage1 / parity check (experiments)")
    ap.add_argument("--chunk", type=int, default=8192, help="keyframes per DB-build batch")
    ap.add_argument("--workload", default="city", choices=["city", "seq"],
                    help="city: configs[3] node-level DB (default, the metric's config); "
                         "seq: configs[1]-shaped labelled-scan sequence, stages 1-4 per query scan")
    ap.add_argument("--shards", type=int, default=0,
                    help="city, N > 1: keyframe-range shards S (default 0 = N: one shard per GPU, the metric's layout). "
                         "S < N: N / S replicas of every shard, each group of S ranks serves its own slice of the query batch")
    ap.add_argument("--scans", type=int, default=1024, help="seq: map keyframes (scans)")
    ap.add_argument("--batch", type=int, default=128, help="seq: query scans per call")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step returned (loop results, candidates, and the match / inlier "
                         "lists of a seeded sample of queries) to DIR/<name>.npy (float64); --impl ours only, the "
                         "reference arm is a CPU comparison and is not dumped.  seq: that step keeps its results "
                         "until they are written, so its later batches take fresh buffers")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    return args


def plan_layout(rank, world, shards, nkf, nq):
    """S keyframe-range shards x R = world / S replica groups.  Group g = ranks g*S .. g*S+S-1 holds the
    whole database once (shard s = keyframes [s*fpr, (s+1)*fpr)) and serves queries [g*nq/R, (g+1)*nq/R).
    shards = 0 means S = world: one shard per GPU, every GPU votes the whole batch (BASELINE.json configs[3])."""
    S = shards if shards > 0 else world
    if world % S:
        raise ValueError("--shards must divide the number of GPUs")
    R = world // S
    grp, srank = rank // S, rank % S
    fpr = (nkf + S - 1) // S
    lo, hi = (srank * fpr, min(nkf, (srank + 1) * fpr)) if S > 1 else (0, nkf)
    return {"S": S, "R": R, "group": grp, "shard_rank": srank, "frames_per_rank": fpr, "frame_lo": lo, "frame_hi": max(hi, lo),
            "query_lo": grp * nq // R, "query_hi": (grp + 1) * nq // R}


# ------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks/throttle reasons DURING the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            if len(r) < 9:
                continue
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
            except ValueError:
                continue
            for n, v in zip(names, r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def source_sha(path="sgtd_b200/csrc/search.cu"):
    return hashlib.sha256(open(os.path.join(ROOT, path), "rb").read()).hexdigest()[:16]


def ncu_traffic(kernel, nkf, nq, world):
    """dram__bytes_read.sum + dram__bytes_write.sum of ONE launch of `kernel`, from the committed record
    tools/ncu_traffic.py writes out of an `ncu --set full` capture of this workload.  Returns
    (bytes or None, provenance)."""
    p = os.path.join(ROOT, "profiles", "r02_traffic.json")
    if not os.path.exists(p):
        return None, "no profiles/r02_traffic.json"
    for rec in json.load(open(p)).get("records", []):
        if rec["kernel"] == kernel and rec["keyframes"] == nkf and rec["queries"] == nq and rec["n_gpus"] == world:
            stale = rec.get("source_sha") != source_sha()
            return rec["dram_read_bytes"] + rec["dram_write_bytes"], {
                "file": "profiles/r02_traffic.json", "report": rec.get("report"), "source_sha": rec.get("source_sha"),
                "captured_kernel_ms": rec.get("duration_ms"), "stale_vs_current_source": stale}
    return None, "no record for this kernel / workload / sharding in profiles/r02_traffic.json"


def result_crc(loops, cands):
    c = 0
    for a in (loops["frame"], loops["score"], cands["frame"], cands["votes"], cands["score"]):
        c = zlib.crc32(np.ascontiguousarray(a).tobytes(), c)
    return c


DUMP_LIMIT_BYTES = 64 << 20
LOOP_FIELDS = ("frame", "ncand", "score")
DUMP_CAND_FIELDS = ("frame", "votes", "nmatch", "score", "ninlier", "best_hyp", "R", "t")
LIST_QUERIES, LIST_CANDS, LIST_LIMIT_BYTES = 64, 4, 16 << 20


def search_lists(parts, cands):
    """Match lists (query descriptor, probe ordinal, DB descriptor) and inlier lists of the first LIST_CANDS
    candidates of a fixed, seeded sample of LIST_QUERIES queries, as a caller fetches them from the results.
    parts: (first query, SearchResult) pairs, ascending, covering the queries of `cands`.  Only candidates this
    rank owns carry lists (sharded databases); inlier lists only for verified candidates (score >= 0).
    Lists stop at LIST_LIMIT_BYTES."""
    nq = cands.shape[0]
    pick = np.sort(np.random.default_rng(1).choice(nq, min(nq, LIST_QUERIES), replace=False))
    key, m, inl, nbytes = [], [], [], 0
    for q in pick:
        q0, res = [p for p in parts if p[0] <= q][-1]
        cq = cands[q]
        for c in np.nonzero((cq["frame"] >= 0) & (cq["match_off"] >= 0))[0][:LIST_CANDS]:
            mq, mc, mg = res.matches(q - q0, int(c), int(cq["nmatch"][c]))
            il = res.inliers(q - q0, int(c), int(cq["ninlier"][c])) if cq["score"][c] >= 0 else np.zeros(0, np.int32)
            nbytes += 8 * (3 * mq.size + il.size + 4)
            if nbytes > LIST_LIMIT_BYTES:
                break
            key.append((q, c)); m.append(np.stack([mq, mc, mg], 1)); inl.append(il)
    key = np.array(key, np.int64).reshape(-1, 2)
    mm = np.concatenate(m) if m else np.zeros((0, 3), np.int64)
    return {"list_query": key[:, 0], "list_cand": key[:, 1],
            "list_match_start": np.cumsum([0] + [len(a) for a in m]),       # lists i: [start[i], start[i+1])
            "match_q": mm[:, 0], "match_cell": mm[:, 1], "match_g": mm[:, 2],
            "list_inlier_start": np.cumsum([0] + [len(a) for a in inl]),
            "inlier": np.concatenate(inl) if inl else np.zeros(0, np.int64)}


def dump_outputs(out_dir, loops, cands, lists):
    """What a caller of the search receives -- loop result and candidate list of every query, plus the lists
    of search_lists() -- as float64 .npy files; integer fields are exact in float64.  Buffer offsets
    (match_off, inlier_off) are left out: they locate lists inside the library's buffers and are not
    results.  Above DUMP_LIMIT_BYTES a fixed, seeded sample of the queries is written; query.npy holds the
    indices of the rows written."""
    nq, k = cands.shape
    row_bytes = 8 * (1 + len(LOOP_FIELDS) + k * sum(int(np.prod(cands.dtype[f].shape)) for f in DUMP_CAND_FIELDS))
    budget = DUMP_LIMIT_BYTES - (64 << 10) - sum(8 * a.size for a in lists.values())   # 64 KB for the .npy headers
    keep = min(nq, budget // row_bytes)
    rows = np.arange(nq) if keep == nq else np.sort(np.random.default_rng(0).choice(nq, keep, replace=False))
    arrays = dict(lists, query=rows)
    arrays.update({f"loop_{f}": loops[f][rows] for f in LOOP_FIELDS})
    arrays.update({f"cand_{f}": cands[f][rows] for f in DUMP_CAND_FIELDS})
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a, np.float64))


def per_probe_model_bytes(st):
    return 32 * st["Q"] + 16 * st["P"] + 28 * st["E"] + 12 * st["M"]


def one_pass_bytes(st, nq, F):
    """What any formulation of the vote stage has to move at least once (see module docstring)."""
    return 16 * st["Eu"] + 32 * st["Q"] + 16 * st["P"] + 4 * nq * F


def se3(pose):
    c, s_ = np.cos(pose[2]), np.sin(pose[2])
    T = np.eye(4)
    T[:2, :2] = [[c, -s_], [s_, c]]
    T[:2, 3] = pose[:2]
    return T


def success_stats(loops, cands, poses, qposes):
    """The reference's success criterion (semantic_graph_localization.cpp:724-750, compute_adj_rpe
    utility.hpp:110-123) through the library's own helper, plus the recall@k bookkeeping (:603-646)."""
    from sgtd_b200 import capi
    nq = loops.shape[0]
    map12 = np.stack([se3(p)[:3].reshape(12) for p in poses])
    found = succ = within = 0
    terr, rerr, ranks = [], [], []
    for qi in range(nq):
        n = int(loops["ncand"][qi])
        gt12 = se3(qposes[qi])[:3].reshape(12)
        if n:
            ranks.append(capi.recall_rank(cands[qi, :n], map12, gt12, 10.0)[0])
        f = loops["frame"][qi]
        if f < 0:
            continue
        found += 1
        within += np.hypot(*(poses[f, :2] - qposes[qi, :2])) < 10.0
        c = [c for c in cands[qi] if c["frame"] == f and c["score"] == loops["score"][qi]][0]
        ok, te, re, _ = capi.localization_check(map12[f], c["R"], c["t"], gt12)
        terr.append(te); rerr.append(re)
        succ += ok
    ranks = np.array(ranks) if ranks else np.zeros(0, int)
    return {"queries": nq, "found": int(found), "within_10m": int(within), "success_T5m_R10deg": int(succ),
            "rmse_t_m": float(np.sqrt(np.mean(np.square(terr)))) if terr else None,
            "rmse_r_deg": float(np.sqrt(np.mean(np.square(rerr)))) if rerr else None,
            "recall_at_1": float(np.mean(ranks == 0)) if ranks.size else None,
            "recall_at_5": float(np.mean((ranks >= 0) & (ranks < 5))) if ranks.size else None,
            "recall_at_50": float(np.mean(ranks >= 0)) if ranks.size else None}


def build_db(mgr, xyz, lab, off, lo, hi, chunk):
    """stage 2 on the GPU for the keyframes [lo, hi) this rank owns; the others only advance frame ids"""
    import numpy as np
    from sgtd_b200 import capi
    nkf = off.shape[0] - 1
    nodes = capi.make_nodes(xyz, lab)
    for c0 in range(0, nkf, chunk):
        c1 = min(nkf, c0 + chunk)
        if c1 <= lo or c0 >= hi:
            b = mgr.upload(np.zeros(0, capi.DESC_DTYPE), np.zeros(c1 - c0 + 1, np.int64))
        else:
            b = mgr.build(nodes, off[c0:c1 + 1], frame_ids=np.arange(c0, c1, dtype=np.uint32))
        mgr.add(b)
        b.free()
    mgr.finalize()


# ------------------------------------------------------------------------------------------
# CPU arms
def cpu_port_sample(cfg, nkf_cpu, nq_cpu, nthreads):
    """Oracle (CPU port of the reference) on a bounded sample: the first nkf_cpu keyframes as DB and
    nq_cpu queries whose true place lies inside that prefix."""
    from oracle import orc
    xyz, lab, off = cfg["db"]
    qx, ql, qo = cfg["queries"]
    nkf = min(nkf_cpu, off.shape[0] - 1)
    o = orc.Oracle()
    t0 = time.time()
    o.build_add_many(xyz[:off[nkf]], lab[:off[nkf]], off[:nkf + 1], nthreads)
    t_build = time.time() - t0
    inside = np.nonzero(cfg["gt"] < nkf)[0]
    pick = inside[:nq_cpu] if inside.size >= nq_cpu else np.arange(nq_cpu)
    t0 = time.time()
    for q in pick:
        qd = o.build(qx[qo[q]:qo[q + 1]], ql[qo[q]:qo[q + 1]])   # BuildSingleScanSTD
        o.search(qd, nthreads=nthreads, want_votes=False)        # SearchLoop
    return len(pick) / (time.time() - t0), nkf, len(pick), t_build


def reference_build_timings(nkf=1000, nq=4, threads=(4, 8)):
    """The reference's own STDesc.cpp (oracle/_ref) and the lean port on the same 1k-keyframe DB
    (configs[0]-sized): the 'reference-faithful' vs 'lean' CPU variants of SURVEY 8d."""
    from oracle import orc, ref
    from sgtd_b200 import synth
    if not ref.available():
        return {"unavailable": "oracle/_ref/libsgtd_ref.so not present"}
    cfg = synth.make_config(0, nkf, nq)
    xyz, lab, off = cfg["db"]
    qx, ql, qo = cfg["queries"]
    r, o = ref.Reference(), orc.Oracle()
    for f in range(nkf):
        r.build(xyz[off[f]:off[f + 1]], lab[off[f]:off[f + 1]])
        r.add_last()
    o.build_add_many(xyz, lab, off)
    out = {"keyframes": nkf, "queries": nq, "db_descriptors": int(o.db_size), "unit": "queries/s"}
    ncpu = os.cpu_count() or 1
    for th in sorted(set(list(threads) + [ncpu])):
        t0 = time.time()
        for q in range(nq):
            r.build(qx[qo[q]:qo[q + 1]], ql[qo[q]:qo[q + 1]])
            r.search(nthreads=th, want_lists=False)
        out[f"reference_{th}_threads"] = nq / (time.time() - t0)
        t0 = time.time()
        for q in range(nq):
            o.search(o.build(qx[qo[q]:qo[q + 1]], ql[qo[q]:qo[q + 1]]), nthreads=th, want_votes=False)
        out[f"port_{th}_threads"] = nq / (time.time() - t0)
    out["note"] = ("reference_*: R/src/STDesc.cpp compiled unmodified (oracle/_ref), OpenMP thread count = MP_PROC_NUM; "
                   "port_*: oracle/sgtd_oracle.cpp, same results with compact records")
    return out


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import orc
    from sgtd_b200 import synth
    ncores = os.cpu_count() or 1
    cfg = synth.make_config(3, args.keyframes, args.queries)
    xyz, lab, off = cfg["db"]
    qx, ql, qo = cfg["queries"]
    nkf, nq = off.shape[0] - 1, qo.shape[0] - 1
    o = orc.Oracle()
    t0 = time.time()
    o.build_add_many(xyz, lab, off, ncores)          # the SAME database as our arm: all keyframes
    t_build = time.time() - t0

    def run_queries(idx):
        for q in idx:
            qd = o.build(qx[qo[q]:qo[q + 1]], ql[qo[q]:qo[q + 1]])
            o.search(qd, nthreads=ncores, want_votes=False)

    t0 = time.time()
    run_queries([0])
    t_q = time.time() - t0
    per_step = int(max(1, min(8, args.ref_budget_s / max(args.steps + args.warmup, 1) / max(t_q, 1e-3))))
    order = np.random.default_rng(0).permutation(nq)
    pos = 0

    def step():
        nonlocal pos
        idx = [order[(pos + i) % nq] for i in range(per_step)]
        pos += per_step
        run_queries(idx)

    for _ in range(args.warmup):
        step()
    t0 = time.time()
    for _ in range(args.steps):
        step()
    dt = time.time() - t0
    v = args.steps * per_step / dt
    sample = (f"{per_step} queries/step against ALL {nkf} keyframes ({o.db_size} descriptors), oracle port with {ncores} "
              f"OpenMP threads; DB build {t_build:.0f}s not timed")
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": "queries/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": WORKLOAD, "keyframes": nkf, "queries": nq, "db_descriptors": int(o.db_size),
                       "sharding": f"keyframe-range x{args.gpus}", "l2": "inputs larger than L2 (DB index >> 126 MB)"},
            "queries_per_step": per_step,
            "cpu_baseline": {"value": v, "unit": "queries/s", "cores": ncores, "kind": "port", "sample": sample},
            "e2e": {"value": v, "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    del o
    try:
        line["reference_build"] = reference_build_timings()
    except Exception as e:  # the headline CPU number above does not depend on it
        line["reference_build"] = {"error": repr(e)}
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------
class Timer:
    """CUDA events on the library's stream, barrier + synchronize on both sides, max over ranks."""

    def __init__(self, torch, dist, dev, world, stream_ptr):
        self.torch, self.dist, self.dev, self.world = torch, dist, dev, world
        self.stream = torch.cuda.ExternalStream(stream_ptr, device=dev)

    def barrier(self):
        self.torch.cuda.synchronize()
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def __call__(self, fn, steps, last=None):
        """times `steps` calls; `last`, when given, is called instead of fn in the final step"""
        e0, e1 = self.torch.cuda.Event(enable_timing=True), self.torch.cuda.Event(enable_timing=True)
        keep = []
        self.barrier()
        e0.record(self.stream)
        for i in range(steps):
            keep.append(last() if last and i == steps - 1 else fn())
        e1.record(self.stream)
        self.barrier()
        ms = e0.elapsed_time(e1)
        if self.world > 1:
            t = self.torch.tensor([ms], device=self.dev)
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms, keep


def sweep_entry(torch, dev, cfg_index, nkf, nq, chunk, peak, steps, warmup):
    """one point of queries/s vs DB size (single GPU, device-resident queries)"""
    from sgtd_b200 import capi, synth
    cfg = synth.make_config(cfg_index, nkf, nq)
    xyz, lab, off = cfg["db"]
    qx, ql, qo = cfg["queries"]
    mgr = capi.STDescManager(device=dev.index)
    build_db(mgr, xyz, lab, off, 0, nkf, chunk)
    q_dev = torch.from_numpy(capi.make_nodes(qx, ql).view(np.uint8).reshape(-1)).to(dev)
    mgr.set_option("stats_unique", 1)
    qb = mgr.build(q_dev.data_ptr(), qo)
    res = mgr.search(qb)
    st_u, _ = res.stats()
    res.free(); qb.free()
    mgr.set_option("stats_unique", 0)

    def step():
        qb = mgr.build(q_dev.data_ptr(), qo)
        res = mgr.search(qb)
        out = res.stats()
        res.free(); qb.free()
        return out

    for _ in range(warmup):
        step()
    timer = Timer(torch, None, dev, 1, mgr.stream)
    ms, kept = timer(step, steps)
    vms = float(np.mean([tm["vote_ms"] for _, tm in kept]))
    bound = one_pass_bytes(st_u, nq, nkf)
    out = {"keyframes": nkf, "queries": nq, "db_descriptors": int(mgr.db_size), "queries_per_s": nq * steps / (ms * 1e-3),
           "ms_per_step": ms / steps, "vote_kernel_ms": vms, "vote_one_pass_gbs": bound / (vms * 1e-3) / 1e9,
           "vote_one_pass_frac": bound / (vms * 1e-3) / 1e9 / peak, "stage_ms": {k: round(float(np.mean([tm[k] for _, tm in kept])), 3)
                                                                                 for k in ("probe_ms", "vote_ms", "topk_ms", "collect_ms", "verify_ms", "total_ms")}}
    mgr.close()
    return out


def stage1_record(torch, dev, peak, steps, warmup, nscans=128):
    """instance extraction (stage 1) on a batch of labelled 64-beam scans of the configs[1]-shaped street
    sequence, scans resident in HBM: scans/s and GB/s on the SURVEY 8d figure of 24 B/point."""
    from sgtd_b200 import capi, synth, synth_seq
    w = synth_seq.make_street_world(4541, synth.BASE_SEED + 1)
    sel = np.linspace(0, 4540, nscans).astype(int)
    pts, labs, off = [], [], [0]
    for i in sel:
        p, l = synth_seq.render_at(w, w["poses"][i], 10_000 + int(i), device=dev)
        pts.append(p); labs.append(l.to(torch.int32)); off.append(off[-1] + p.shape[0])
    pts, labs, off = torch.cat(pts).contiguous(), torch.cat(labs).contiguous(), np.array(off, np.int64)
    mgr = capi.STDescManager(device=dev.index)

    def step():
        return mgr.extract_instances_ptr(pts.data_ptr(), labs.data_ptr(), off)

    for _ in range(warmup):
        step()
    l0 = mgr.kernel_launches
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(steps):
        nodes, noff, ninst = step()
    torch.cuda.synchronize()
    ms = (time.perf_counter() - t0) * 1e3 / steps
    npts = int(off[-1])
    gbs = 24.0 * npts / (ms * 1e-3) / 1e9
    out = {"scans": nscans, "points": npts, "points_per_scan": npts // nscans, "nodes_per_scan": float(np.diff(noff).mean()),
           "ms_per_batch": ms, "scans_per_s": nscans / (ms * 1e-3), "algorithmic_bytes_per_point": 24,
           "achieved_gbs": gbs, "frac_of_hbm_peak": gbs / peak, "gpu_launches_per_batch": int((mgr.kernel_launches - l0) / steps),
           "timing": "wall clock around the synchronous C-ABI call (device work + the host-side part of the call)"}
    tm = mgr.stage1_timings() if hasattr(mgr, "stage1_timings") else None
    if tm:
        out["device_ms"] = tm
    mgr.close()
    return out


def run_ours(args):
    import torch
    import torch.distributed as dist
    from sgtd_b200 import capi, synth

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    cfg = synth.make_config(3, args.keyframes, args.queries)
    xyz, lab, off = cfg["db"]
    qx, ql, qo = cfg["queries"]
    nkf = off.shape[0] - 1
    nq = qo.shape[0] - 1

    mgr = capi.STDescManager(device=local)
    # layout: S keyframe-range shards x R = N / S replicas; replica group g (ranks g*S .. g*S+S-1) serves
    # queries [g*nq/R, (g+1)*nq/R) against its own copy of the S shards.  Default S = N (R = 1): every GPU
    # holds one shard and votes the whole batch (BASELINE.json configs[3]).
    L = plan_layout(rank, world, args.shards, nkf, nq)
    S, R, grp, srank, fpr = L["S"], L["R"], L["group"], L["shard_rank"], L["frames_per_rank"]
    if S > 1:
        mine = torch.from_numpy(capi.nccl_unique_id()).to(dev)
        ids = [torch.zeros_like(mine) for _ in range(world)]
        dist.all_gather(ids, mine)                 # the id of a group is its leader's
        mgr.shard_init(srank, S, fpr, ids[grp * S].cpu().numpy())
    lo, hi = L["frame_lo"], L["frame_hi"]
    q0, q1, nq_all = L["query_lo"], L["query_hi"], nq
    if R > 1:
        qx, ql = qx[qo[q0]:qo[q1]], ql[qo[q0]:qo[q1]]
        qo = (qo[q0:q1 + 1] - qo[q0]).astype(np.int64)
        nq = q1 - q0

    # ---- database build (not timed): stage 2 on the GPU for this rank's keyframes ----
    t0 = time.time()
    build_db(mgr, xyz, lab, off, lo, hi, args.chunk)
    t_db = time.time() - t0
    assert mgr.current_frame_id_ == nkf

    # ---- inputs: query nodes in HBM (value) and in pinned host memory (e2e) ----
    qnodes = capi.make_nodes(qx, ql)
    q_dev = torch.from_numpy(qnodes.view(np.uint8).reshape(-1)).to(dev)
    q_pin = torch.from_numpy(qnodes.view(np.uint8).reshape(-1).copy()).pin_memory()
    q_pin_np = q_pin.numpy().view(capi.NODE_DTYPE)
    k = mgr.cfg.candidate_num
    loops_pin = torch.empty(nq * capi.LOOP_DTYPE.itemsize, dtype=torch.uint8).pin_memory()
    cands_pin = torch.empty(nq * k * capi.CAND_DTYPE.itemsize, dtype=torch.uint8).pin_memory()

    held = []                                     # --dump-outputs: the search of the last timed step

    def step_device(keep=False):
        qb = mgr.build(q_dev.data_ptr(), qo)
        res = mgr.search(qb)
        out = res.stats()
        if keep:
            held[:] = [res, qb]
        else:
            res.free(); qb.free()                 # buffers go back to the handle's pool
        return out

    def step_e2e():
        qb = mgr.build(q_pin_np, qo)              # H2D of the node arrays inside
        res = mgr.search(qb)
        capi.lib().sgtd_result_download(mgr._h, res.ptr, ctypes.c_void_p(loops_pin.data_ptr()),
                                        ctypes.c_void_p(cands_pin.data_ptr()))   # D2H
        out = res.stats()
        res.free(); qb.free()
        return out

    timer = Timer(torch, dist, dev, world, mgr.stream)

    # ---- warm-up; one of the warm-up steps doubles as the parity check: the exact FP64 streaming
    # kernel must give byte-identical vote rows and candidates (this rank's shard) ----
    F_local = hi - lo
    parity = None
    if not args.no_extras:
        def digest(stream_mode):
            mgr.set_option("vote_stream", 1 if stream_mode else 0)
            mgr.set_option("stats_unique", 0 if stream_mode else 1)
            qb = mgr.build(q_dev.data_ptr(), qo)
            res = mgr.search(qb)
            c = 0
            for q in range(nq):
                c = zlib.crc32(res.votes(q, F_local).tobytes(), c)
            lp, cd = res.download()
            st, _ = res.stats()
            res.free(); qb.free()
            return (c, zlib.crc32(lp.tobytes()), zlib.crc32(cd.tobytes())), st
        d_join, st_unique = digest(False)
        d_stream, _ = digest(True)
        mgr.set_option("vote_stream", 0)
        mgr.set_option("stats_unique", 0)
        parity = d_join == d_stream
        if world > 1:
            t = torch.tensor([int(parity)], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MIN)
            parity = bool(t.item())
        assert parity, "vote join and exact streaming kernel disagree"
    else:
        st_unique = None
    for _ in range(args.warmup):
        step_device()
        step_e2e()

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    l0 = mgr.kernel_launches
    ms_dev, kept = timer(step_device, args.steps, last=(lambda: step_device(keep=True)) if args.dump_outputs else None)
    launches = mgr.kernel_launches - l0
    if held:
        loops_dump, cands_dump = held[0].download()
        lists_dump = search_lists([(0, held[0])], cands_dump) if rank == 0 else None   # rank 0 serves queries from 0
        for b in held:
            b.free()
    # per-kernel numbers from the timed steps themselves (events recorded inside the library)
    vote_ms, stats, stage = [], None, {}
    for st, tm in kept:
        vote_ms.append(tm["vote_ms"]); stats = st
        for kk, vv in tm.items():
            stage[kk] = stage.get(kk, 0.0) + vv / len(kept)
    # shards differ (database density, where the batch's candidates fall): slowest / fastest rank per stage
    stage_spread = None
    if world > 1:
        keys = [kk for kk in ("probe_ms", "vote_ms", "topk_ms", "exchange_ms", "collect_ms", "verify_ms", "total_ms") if kk in stage]
        tmax = torch.tensor([stage[kk] for kk in keys], device=dev, dtype=torch.float64)
        tmin = tmax.clone()
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        dist.all_reduce(tmin, op=dist.ReduceOp.MIN)
        stage_spread = {kk: [round(float(a), 3), round(float(b), 3)] for kk, a, b in zip(keys, tmin.tolist(), tmax.tolist())}
    ms_e2e, kept = timer(step_e2e, args.steps)
    loops = np.frombuffer(loops_pin.numpy().tobytes(), capi.LOOP_DTYPE)
    cands_h = np.frombuffer(cands_pin.numpy().tobytes(), capi.CAND_DTYPE).reshape(nq, k)
    if R > 1:
        # the replica groups' slices of the batch, in query order, for the checksum and the success statistics
        # (every rank of a group holds the group's results; equal slice sizes are required here)
        assert nq_all % R == 0, "--shards: the query batch must split evenly over the replica groups"
        def gather(a):
            t = torch.from_numpy(np.frombuffer(a.tobytes(), np.uint8).copy()).to(dev)
            parts = [torch.zeros_like(t) for _ in range(world)]
            dist.all_gather(parts, t)
            return np.concatenate([parts[g * S].cpu().numpy() for g in range(R)])
        loops = np.frombuffer(gather(loops).tobytes(), capi.LOOP_DTYPE)
        cands_h = np.frombuffer(gather(cands_h).tobytes(), capi.CAND_DTYPE).reshape(nq_all, k)
        if args.dump_outputs:
            loops_dump = np.frombuffer(gather(loops_dump).tobytes(), capi.LOOP_DTYPE)
            cands_dump = np.frombuffer(gather(cands_dump).tobytes(), capi.CAND_DTYPE).reshape(nq_all, k)
    clocks = sampler.stop() if rank == 0 else None
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, loops_dump, cands_dump, lists_dump)

    if rank == 0:
        peak, peak_src = measured_peak()
        vms = float(np.mean(vote_ms))
        vote_kernel = "k_vote_join"
        traffic, traffic_src = ncu_traffic(vote_kernel, nkf, nq, world)
        roof = {"bound": "hbm", "kernel": vote_kernel, "peak": peak, "unit": "GB/s", "peak_source": peak_src,
                "peak_nominal": 8000.0, "avg_launch_ms": vms, "traffic": traffic, "traffic_source": traffic_src,
                "counters": stats, "per_probe_model_bytes": per_probe_model_bytes(stats),
                "per_probe_model_gbs": per_probe_model_bytes(stats) / (vms * 1e-3) / 1e9}
        if st_unique is not None and "Eu" in st_unique:
            bound = one_pass_bytes(st_unique, nq, F_local)      # this rank's kernel, this rank's bytes
            ach = bound / (vms * 1e-3) / 1e9
            roof.update({"achieved": ach, "frac": ach / peak, "frac_nominal": ach / 8000.0,
                         "algorithmic_bytes_per_launch": bound, "distinct_buckets": st_unique["B"],
                         "distinct_bucket_entries": st_unique["Eu"],
                         "reread_factor": (traffic / bound) if traffic else None,
                         "traffic_gbs": (traffic / (vms * 1e-3) / 1e9) if traffic else None,
                         "traffic_frac_of_peak": (traffic / (vms * 1e-3) / 1e9 / peak) if traffic else None,
                         "votes_per_s": stats["M"] / (vms * 1e-3),
                         "note": "achieved = one-pass bound (16 B x entries of the distinct probed buckets + 32 B x query "
                                 "descriptors + 16 B x probes + 4 B x vote cells) / CUDA-event time of the vote kernel; "
                                 "traffic = ncu DRAM bytes of one launch (profiles/r02_traffic.json); the kernel casts M "
                                 "vote increments (RED) per launch -- see DESIGN.md section 4 for what bounds it"})
        else:
            roof.update({"achieved": None, "frac": None})
        line = {
            "metric": METRIC, "value": nq_all * args.steps / (ms_dev * 1e-3), "unit": "queries/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_dev / args.steps,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": WORKLOAD, "keyframes": nkf, "queries": nq_all, "db_descriptors": None,
                       "sharding": f"keyframe-range x{S}" + (f", {R} replicas of every shard, one slice of the batch per replica group" if R > 1 else ""),
                       "l2": "inputs larger than L2 (DB index >> 126 MB)"},
            "db_build_s": round(t_db, 2),
            "e2e": {"value": nq_all * args.steps / (ms_e2e * 1e-3), "unit": "queries/s",
                    "h2d_bytes_per_step": int(qnodes.nbytes + qo.nbytes) * R,
                    "d2h_bytes_per_step": int(loops_pin.numel() + cands_pin.numel()) * R},
            "gpu_launches": int(launches),
            "parity_checked": parity,
            "roofline": roof,
            "stage_ms": {kk: round(vv, 3) for kk, vv in stage.items()},
            "stage_ms_min_max_over_ranks": stage_spread,
            "recall": success_stats(loops, cands_h, cfg["world"]["poses"], cfg["qposes"]),
            # checksum of (best frame, score, candidate frames/votes/scores): identical for every N
            "result_crc": result_crc(loops, cands_h.reshape(-1)),
            "clocks": clocks,
        }
    db_total = int(mgr.db_size)
    if world > 1:
        t = torch.tensor([db_total], device=dev, dtype=torch.int64)
        dist.all_reduce(t)
        db_total = int(t.item()) // R              # every replica group holds the whole database once
        dist.barrier()
    mgr.close()
    del mgr
    if rank == 0:
        line["config"]["db_descriptors"] = db_total
        if world == 1 and not args.no_extras:
            sweep = []
            for (ci, skf, snq) in ((0, 1000, 256), (2, 10000, 256)):
                sweep.append(sweep_entry(torch, dev, ci, skf, snq, args.chunk, peak, args.steps, args.warmup))
            sweep.append({"keyframes": nkf, "queries": nq, "db_descriptors": line["config"]["db_descriptors"],
                          "queries_per_s": line["value"], "ms_per_step": line["ms_per_step"], "vote_kernel_ms": vms,
                          "vote_one_pass_gbs": roof.get("achieved"), "vote_one_pass_frac": roof.get("frac"),
                          "stage_ms": line["stage_ms"]})
            line["db_sweep"] = sweep
            line["stage1"] = stage1_record(torch, dev, peak, args.steps, args.warmup)
        if not args.no_cpu_baseline:
            ncores = os.cpu_count() or 1
            v, nk, npick, tb = cpu_port_sample(cfg, args.cpu_keyframes, args.cpu_queries, ncores)
            line["cpu_baseline"] = {
                "value": v, "unit": "queries/s", "cores": ncores, "kind": "port",
                "sample": f"{npick} queries against the first {nk} of {nkf} keyframes, oracle with {ncores} OpenMP threads "
                          f"(bounded sample: CPU cost grows with DB size, so it favours the CPU; --impl reference runs the full DB)"}
            if world == 1 and not args.no_extras:
                try:
                    line["cpu_baseline"]["reference_build"] = reference_build_timings()
                except Exception as e:
                    line["cpu_baseline"]["reference_build"] = {"error": repr(e)}
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


# ------------------------------------------------------------------------------------------
def run_seq(args):
    """configs[1]-shaped workload: a synthetic street sequence of labelled 64-beam scans.  The map is
    built from scans (stage 1 -> stage 2 -> add); every query is a labelled SCAN of a revisited place
    (new noise, lateral offset, random yaw) pushed through stages 1-4.  Single GPU."""
    import torch
    from sgtd_b200 import capi, synth_seq, synth
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(0)
    w = synth_seq.make_street_world(args.scans, synth.BASE_SEED + 1)
    P = w["poses"]
    mgr = capi.STDescManager(device=0)
    nq = min(args.queries, 256) if args.queries == 1024 else args.queries
    B = args.batch

    def render_batch(poses, seed0):
        pts, labs, off = [], [], [0]
        for i, ps in enumerate(poses):
            p, l = synth_seq.render_at(w, ps, seed0 + i, device=dev)
            pts.append(p); labs.append(l.to(torch.int32)); off.append(off[-1] + p.shape[0])
        return torch.cat(pts).contiguous(), torch.cat(labs).contiguous(), np.array(off, np.int64)

    # ---- map pass (not timed): every scan becomes a keyframe; a scan with fewer nodes than
    # descriptor_near_num keeps its frame id and contributes no descriptor (library behaviour) ----
    t0 = time.time()
    few = 0
    for c0 in range(0, args.scans, B):
        pts, labs, off = render_batch(P[c0:c0 + B], 10_000 + c0)
        nodes, noff, _ = mgr.extract_instances_ptr(pts.data_ptr(), labs.data_ptr(), off)
        few += int((np.diff(noff) < mgr.cfg.descriptor_near_num).sum())
        b = mgr.build(nodes, noff, frame_ids=np.arange(c0, c0 + len(off) - 1, dtype=np.uint32))
        mgr.add(b); b.free()
    mgr.finalize()
    t_map = time.time() - t0
    # ---- queries: revisited places, new noise, +-1.5 m lateral offset, random yaw ----
    rng = np.random.default_rng(synth.BASE_SEED + 2)
    gt = rng.integers(0, args.scans, nq)
    qposes = P[gt].copy()
    qposes[:, :2] += rng.uniform(-1.5, 1.5, (nq, 2))
    qposes[:, 2] = rng.uniform(-np.pi, np.pi, nq)
    batches = []
    for c0 in range(0, nq, B):
        pts, labs, off = render_batch(qposes[c0:c0 + B], 900_000 + c0)
        batches.append((pts, labs, off, pts.cpu().pin_memory(), labs.cpu().pin_memory()))
    k = mgr.cfg.candidate_num
    out_loops = np.zeros(nq, capi.LOOP_DTYPE)
    out_cands = np.zeros((nq, k), capi.CAND_DTYPE)
    stage = {}
    held = []                                    # --dump-outputs: (first query, result, batch) of the last timed step

    def step(host, keep=False):
        c0 = 0
        for (pts, labs, off, hp, hl) in batches:
            t = [time.perf_counter()]
            if host:
                nodes, noff, _, _ = mgr.extract_instances(hp.numpy(), hl.numpy().view(np.uint32), off, want_membership=False)
            else:
                nodes, noff, _ = mgr.extract_instances_ptr(pts.data_ptr(), labs.data_ptr(), off)
            t.append(time.perf_counter())
            qb = mgr.build(nodes, noff)          # sparse scans yield no descriptors -> "No STDescs!" -> (-1, 0)
            t.append(time.perf_counter())
            res = mgr.search(qb)
            loops, cands = res.download()
            t.append(time.perf_counter())
            n = len(off) - 1
            out_loops[c0:c0 + n] = loops; out_cands[c0:c0 + n] = cands
            if keep:
                held.append((c0, res, qb))
            else:
                res.free(); qb.free()
            c0 += n
            for name, a, b_ in (("stage1_ms", 0, 1), ("stage2_ms", 1, 2), ("stage34_ms", 2, 3)):
                stage[name] = stage.get(name, 0.0) + (t[b_] - t[a]) * 1e3

    def timed(host, steps, keep_last=False):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for i in range(steps):
            step(host, keep_last and i == steps - 1)
        torch.cuda.synchronize()
        return (time.perf_counter() - t0) * 1e3

    for _ in range(args.warmup):
        step(False); step(True)
    sampler = ClockSampler(0)
    sampler.start()
    stage.clear()
    l0 = mgr.kernel_launches
    ms_dev = timed(False, args.steps, keep_last=bool(args.dump_outputs))
    launches = mgr.kernel_launches - l0
    if args.dump_outputs:                        # step() leaves the last timed step's results in out_*
        dump_outputs(args.dump_outputs, out_loops, out_cands, search_lists([(c0, res) for c0, res, _ in held], out_cands))
        for _, res, qb in held:
            res.free(); qb.free()
    st_dev = {kk: round(vv / args.steps, 2) for kk, vv in stage.items()}
    ms_e2e = timed(True, args.steps)
    clocks = sampler.stop()
    npts = int(sum(b[2][-1] for b in batches))
    peak, _ = measured_peak()
    line = {"metric": METRIC, "value": nq * args.steps / (ms_dev * 1e-3), "unit": "queries/s", "n_gpus": 1,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_dev / args.steps, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": "configs[1]-shaped: synthetic street sequence, labelled 64-beam scans, stages 1-4 per query",
                       "map_scans": args.scans, "queries": nq, "points_per_scan": npts // nq, "batch": B,
                       "db_descriptors": int(mgr.db_size), "map_build_s": round(t_map, 1), "map_scans_with_too_few_nodes": few,
                       "timing": "wall clock around synchronous C-ABI calls (device work is synchronised inside each call)"},
            "e2e": {"value": nq * args.steps / (ms_e2e * 1e-3), "unit": "queries/s",
                    "h2d_bytes_per_step": npts * 20, "d2h_bytes_per_step": int(nq * (16 + k * 136))},
            "gpu_launches": int(launches), "stage_ms_per_step": st_dev,
            "stage1": {"scans_per_s": nq / (st_dev["stage1_ms"] * 1e-3), "achieved_gbs": 24.0 * npts / (st_dev["stage1_ms"] * 1e-3) / 1e9,
                       "frac_of_hbm_peak": 24.0 * npts / (st_dev["stage1_ms"] * 1e-3) / 1e9 / peak},
            "recall": success_stats(out_loops, out_cands, P, qposes),
            "clocks": clocks}
    if not args.no_cpu_baseline:
        from oracle import orc
        o = orc.Oracle()
        # the oracle DB is built from the oracle's own stage 1+2 on a bounded prefix of the map
        nmap = min(args.scans, 64)
        for f in range(nmap):
            p_, l_ = synth_seq.render_at(w, P[f], 10_000 + (f // B) * B + f % B, device="cpu")
            r = orc.extract_instances(p_.numpy(), l_.numpy().astype(np.uint32))
            o.add(o.build(r["node_xyz"], r["node_label"]) if len(r["node_label"]) >= 10 else np.zeros(0, orc.DESC_DTYPE))
        pts, labs, off, hp, hl = batches[0]
        n_cpu = min(8, len(off) - 1)
        t0 = time.time()
        for s in range(n_cpu):
            r = orc.extract_instances(hp.numpy()[off[s]:off[s + 1]], hl.numpy().view(np.uint32)[off[s]:off[s + 1]])
            if len(r["node_label"]) >= 10:
                o.search(o.build(r["node_xyz"], r["node_label"]), nthreads=os.cpu_count() or 1, want_votes=False)
        line["cpu_baseline"] = {"value": n_cpu / (time.time() - t0), "unit": "queries/s", "cores": os.cpu_count() or 1,
                                "kind": "port", "sample": f"{n_cpu} query scans, stages 1-4, against the first {nmap} map scans"}
    print(json.dumps(line))
    mgr.close()


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    elif a.workload == "seq":
        run_seq(a)
    else:
        run_ours(a)
