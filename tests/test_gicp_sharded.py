"""GICP refinement on keyframe-range shards: sgtd_gicp_refine_batch on a handle with a communicator.

CPU part: the workload generator produces what the GPU cases rely on (ownership spread over every rank,
a query wholly on the open-ended last range, an idle rank, skipped candidates, an empty query).
GPU part: without a communicator a virtual shard behaves as an unsharded handle; with one (2 and 4
devices), every rank returns the unsharded handle's outputs bit for bit, whatever the store holds beyond
the rank's own range, the wave size, the visit order or where the sources live; waves match the unsharded
call's and the problems split over the ranks by keyframe ownership; and an invalid call fails on every rank
alike, leaving the group usable."""
import queue
import traceback

import numpy as np
import pytest

from test_gicp import motion, scene

F32 = np.float32
FPR = 3                                   # frames per rank
NQ, STRIDE = 10, 9
BEST = [15.0, 0.5, 1e-9]
WAVES = [0, 1, 3]
CHILD_TIMEOUT = 600


def owner(f, nranks):
    """rank owning keyframe f under sgtd_shard_init's ranges (the last one open-ended)"""
    return min(int(f) // FPR, nranks - 1)


def sharded_batch(nranks, idle_rank=None, n_s=500, n_t=1500, seed=0):
    """Keyframes 0 .. nranks*FPR+1 (the last two beyond nranks*FPR, in the last rank's open range), frames 1 and
    FPR+1 without a cloud, and NQ query sources seen from near a keyframe with a known motion.  Query 0's
    candidates lie one on every rank, query 1's all on the last rank, query 2 has none, the others mix the
    right keyframe, other keyframes, frame -1 and cloudless frames.  idle_rank: that rank's candidates are
    moved to rank 0's frames, so it owns none."""
    from sgtd_b200 import capi
    rng = np.random.default_rng(seed)
    nkf = nranks * FPR + 2
    missing = {1, FPR + 1}
    tgts = {f: scene(np.random.default_rng(1000 + f), n_t) * F32(1.0 + 0.15 * (f % 4)) + F32(3 * f)
            for f in range(nkf) if f not in missing}
    with_cloud = sorted(tgts)
    cands, nc, srcs = np.zeros((NQ, STRIDE), capi.CAND_DTYPE), np.zeros(NQ, np.int32), []
    for q in range(NQ):
        if q == 0:
            fr = [r * FPR + 2 for r in range(nranks)][:STRIDE - 1] + [-1]
        elif q == 1:
            fr = [(nranks - 1) * FPR, nranks * FPR + 1, nranks * FPR, (nranks - 1) * FPR + 2]
        elif q == 2:
            fr = []
        else:
            g = int(rng.choice(with_cloud))
            fr = [g, int(rng.choice(with_cloud)), -1, int(rng.choice(sorted(missing))), int(rng.choice(with_cloud)), g]
            fr = [fr[i] for i in rng.permutation(len(fr))][:4 + q % 3]
        g = next((f for f in fr if f in tgts), with_cloud[q % len(with_cloud)])
        R, t = motion(rng, 2.0, (0.3, -0.2, 0.04))
        pts = tgts[g][rng.choice(n_t, n_s, replace=False)] + rng.normal(0, 0.01, (n_s, 3))
        srcs.append(((pts - t) @ R).astype(F32))
        nc[q] = len(fr)
        for c, f in enumerate(fr):
            if idle_rank is not None and f >= 0 and owner(f, nranks) == idle_rank:
                f %= FPR
            Ri, ti = motion(rng, 1.0, t + rng.normal(0, 0.05, 3))
            cands["frame"][q, c], cands["score"][q, c] = f, rng.integers(0, 50)
            cands["R"][q, c], cands["t"][q, c] = Ri.reshape(9), ti
    off = np.concatenate([[0], np.cumsum([len(s) for s in srcs])]).astype(np.int64)
    order = np.argsort(-cands["score"], axis=1, kind="stable").astype(np.int32)
    return dict(nranks=nranks, nkf=nkf, tgts=tgts, srcs=srcs, src=np.concatenate(srcs), off=off, cands=cands,
                ncand=nc, order=order)


def add_clouds(mgr, B, frames, prm):
    frames = [f for f in sorted(frames) if f in B["tgts"]]
    if frames:
        cl = [B["tgts"][f] for f in frames]
        off = np.concatenate([[0], np.cumsum([len(c) for c in cl])]).astype(np.int64)
        mgr.gicp_map_add(np.concatenate(cl), off, frame_ids=np.array(frames), params=prm)


def own_frames(B, rank):
    return [f for f in B["tgts"] if owner(f, B["nranks"]) == rank]


def expected_problems(B, nal, wave, rank):
    """problems rank aligns: per query, the held candidates (in visit order) of every wave up to the one
    that holds the query's stopping point (n_aligned), counted where rank owns the frame"""
    n = 0
    for q in range(NQ):
        k = int(B["ncand"][q])
        vis = [B["cands"]["frame"][q, c] for c in (B["order"][q, :k] if B["use_order"] else range(k))]
        vis = [f for f in vis if f in B["tgts"]]
        end, w = 0, 0
        while end < nal[q]:                   # a query with a held candidate aligns at least one (nal >= 1)
            end += wave if wave else 1 << w
            w += 1
        n += sum(1 for f in vis[:end] if owner(f, B["nranks"]) == rank)
    return n


# ---- CPU: the workload is what the GPU cases claim -------------------------------------------------------
@pytest.mark.parametrize("nranks", [2, 4, 8])
def test_sharded_workload_shape(nranks):
    B = sharded_batch(nranks)
    fr, nc = B["cands"]["frame"], B["ncand"]
    own = lambda q: {owner(f, nranks) for f in fr[q, :nc[q]] if f >= 0}
    assert own(0) == set(range(nranks))                                       # spread over every rank
    assert own(1) == {nranks - 1} and (fr[1, :nc[1]] >= nranks * FPR).any()   # all on the open-ended last range
    assert nc[2] == 0
    used = [f for q in range(NQ) for f in fr[q, :nc[q]]]
    assert -1 in used and any(f >= 0 and f not in B["tgts"] for f in used)   # skipped candidates
    assert B["nkf"] % FPR != 0 and max(B["tgts"]) >= nranks * FPR
    I = sharded_batch(nranks, idle_rank=1)
    busy = {owner(f, nranks) for q in range(NQ) for f in I["cands"]["frame"][q, :I["ncand"][q]] if f >= 0}
    assert 1 not in busy and busy                                             # an idle rank
    assert I["src"].tobytes() == B["src"].tobytes()


def test_expected_problems_counts_waves():
    B = dict(sharded_batch(2), use_order=False)
    B["ncand"] = np.zeros(NQ, np.int32)
    B["ncand"][1] = 4                                     # frames 3, 7, 6, 5: all held, all on rank 1
    nal = np.zeros(NQ, np.int32)
    for stop, wave, exp in [(1, 0, 1), (2, 0, 3), (4, 0, 4), (2, 1, 2), (2, 3, 3), (4, 3, 4)]:
        nal[1] = stop
        assert expected_problems(B, nal, wave, 1) == exp and expected_problems(B, nal, wave, 0) == 0


# ---- GPU ------------------------------------------------------------------------------------------------
def cases(B):
    for bf in BEST:
        for wave in WAVES:
            for use_order in (True, False):
                yield (bf, wave, use_order)


def run_case(mgr, B, sources, case, k=20):
    bf, wave, use_order = case
    prm = mgr.gicp_params(num_neighbors=k, max_iterations=10, best_fitness=bf)
    mgr.set_option("gicp_wave", wave)
    out = mgr.gicp_refine_batch(sources, B["off"], B["cands"], B["ncand"], B["order"] if use_order else None, prm)
    return tuple(np.ascontiguousarray(a) for a in out) + (mgr.gicp_refine_stats(),)


def same_outputs(a, b):
    return all(x.tobytes() == y.tobytes() for x, y in zip(a[:4], b[:4]))


@pytest.mark.gpu
def test_gpu_virtual_shard_is_unchanged():
    """nranks > 1 without an NCCL id: the store is looked up as on an unsharded handle, clouds outside the
    rank's range included."""
    from sgtd_b200 import capi
    B = sharded_batch(4)
    held = own_frames(B, 1) + [0, 2, 12, 13]
    virt, plain = capi.STDescManager(device=0), capi.STDescManager(device=0)
    try:
        virt.shard_init(1, 4, FPR, None)
        for m in (virt, plain):
            add_clouds(m, B, held, m.gicp_params())
        for case in cases(B):
            a, b = run_case(virt, B, B["src"], case), run_case(plain, B, B["src"], case)
            assert same_outputs(a, b) and a[4] == b[4], case
            assert (a[3] > 0).any()
    finally:
        virt.close(); plain.close()


def _rank_main(rank, nranks, uid, q):
    """one rank of the group: every call below is collective, so each rank makes the same calls in order"""
    try:
        import torch
        from sgtd_b200 import capi
        torch.cuda.set_device(rank)
        mgr = capi.STDescManager(device=rank)
        mgr.shard_init(rank, nranks, FPR, uid)
        B, I = sharded_batch(nranks), sharded_batch(nranks, idle_rank=1)
        prm = mgr.gicp_params()
        d_src = torch.from_numpy(B["src"]).cuda(rank)
        res = {}
        for store in ("own", "all"):
            mgr.gicp_map_clear()
            add_clouds(mgr, B, own_frames(B, rank) if store == "own" else list(B["tgts"]), prm)
            for where, sources in (("host", B["src"]), ("device", d_src.data_ptr())):
                for case in cases(B):
                    res[("main", store, where) + case] = run_case(mgr, B, sources, case)
        res["idle"] = run_case(mgr, I, I["src"], (0.5, 0, True))
        errs = {}
        # one rank's owned clouds stored with another num_neighbors: only that rank can tell, every rank fails
        mgr.gicp_map_clear()
        add_clouds(mgr, B, own_frames(B, rank), mgr.gicp_params(num_neighbors=12 if rank == 1 else 20))
        try:
            run_case(mgr, B, B["src"], (0.5, 0, True))
            errs["k"] = capi.OK
        except capi.SgtdError as e:
            errs["k"] = e.status
        # a source smaller than num_neighbors on query 1, whose candidates only the last rank holds
        mgr.gicp_map_clear()
        add_clouds(mgr, B, own_frames(B, rank), prm)
        small = dict(B, off=B["off"].copy())
        small["off"][2:] -= B["off"][2] - B["off"][1] - 5
        src_small = np.concatenate([B["srcs"][0], B["srcs"][1][:5]] + B["srcs"][2:])
        try:
            run_case(mgr, small, src_small, (0.5, 0, True))
            errs["source"] = capi.OK
        except capi.SgtdError as e:
            errs["source"] = e.status
        res["after_errors"] = run_case(mgr, B, B["src"], (1e-9, 0, True))    # the group still works
        mgr.close()
        q.put((rank, "ok", res, errs))
    except Exception:
        q.put((rank, "error", traceback.format_exc(), None))


def reference(B, I):
    """the unsharded handle on device 0, holding every cloud"""
    from sgtd_b200 import capi
    mgr = capi.STDescManager(device=0)
    try:
        add_clouds(mgr, B, list(B["tgts"]), mgr.gicp_params())
        ref = {case: run_case(mgr, B, B["src"], case) for case in cases(B)}
        ref["idle"] = run_case(mgr, I, I["src"], (0.5, 0, True))
        small = dict(B, off=B["off"].copy())
        small["off"][2:] -= B["off"][2] - B["off"][1] - 5
        with pytest.raises(capi.SgtdError) as e:
            run_case(mgr, small, np.concatenate([B["srcs"][0], B["srcs"][1][:5]] + B["srcs"][2:]), (0.5, 0, True))
        assert e.value.status == capi.E_INVALID
        return ref
    finally:
        mgr.close()


def device_count():
    import torch
    return torch.cuda.device_count() if torch.cuda.is_available() else 0


@pytest.mark.gpu
@pytest.mark.parametrize("nranks", [2, 4])
def test_gpu_sharded_refine_equals_unsharded(nranks):
    import multiprocessing as mp
    from sgtd_b200 import capi
    ndev = device_count()
    print(f"test_gpu_sharded_refine_equals_unsharded: {ndev} CUDA device(s) visible")
    if ndev < nranks:
        pytest.skip(f"{nranks} ranks need {nranks} CUDA devices, {ndev} visible")
    uid = capi.nccl_unique_id()                      # NCCL missing: a failure, not a skip
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_rank_main, args=(r, nranks, uid, q)) for r in range(nranks)]
    try:
        for p in procs:
            p.start()
        B, I = sharded_batch(nranks), sharded_batch(nranks, idle_rank=1)
        ref = reference(B, I)
        got = {}
        for _ in range(nranks):
            try:
                rank, status, res, errs = q.get(timeout=CHILD_TIMEOUT)
            except queue.Empty:
                pytest.fail(f"ranks {sorted(set(range(nranks)) - set(got))} sent nothing within {CHILD_TIMEOUT} s")
            assert status == "ok", f"rank {rank}:\n{res}"
            got[rank] = (res, errs)
        for p in procs:
            p.join(timeout=60)
            assert p.exitcode == 0
    finally:
        for p in procs:
            if p.is_alive():
                p.terminate()
                p.join(timeout=10)
    for rank, (res, errs) in got.items():
        assert errs == {"k": capi.E_INVALID, "source": capi.E_INVALID}, (rank, errs)
        assert same_outputs(res["after_errors"], ref[(1e-9, 0, True)]), rank
        assert same_outputs(res["idle"], ref["idle"]) and res["idle"][4][1] == ref["idle"][4][1], rank
        if rank == 1:
            assert res["idle"][4][0] == 0 and res["idle"][4][2] == 0       # no problem, no round
    for key in got[0][0]:
        if not isinstance(key, tuple):
            continue
        case = key[3:]
        r = ref[case]
        bf, wave, use_order = case
        for rank in got:
            g = got[rank][0][key]
            assert same_outputs(g, r), (rank, key)
            assert g[4][1] == r[4][1], (rank, key, "waves")
            assert g[4][0] == expected_problems(dict(B, use_order=use_order), r[3], wave, rank), (rank, key)
        assert sum(got[rank][0][key][4][0] for rank in got) == r[4][0], key
