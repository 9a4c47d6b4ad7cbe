"""Batched GICP refinement against stored keyframe clouds (sgtd_gicp_map_add / _map_nearest /
_refine_batch).

CPU part: the crafted nearest-neighbour cases land where intended (checked in numpy float32 with
the ((dx*dx)+dy*dy)+dz*dz order), and the workload helpers of tools/bench_gicp.py run at a tiny size.
GPU part: the grid search equals a numpy brute force index for index and bit for bit at several cell
sizes; the batch equals a loop of sgtd_gicp_refine_candidates bit for bit, whatever the wave size and
however its problems are split; a sample agrees with the CPU oracle within test_gicp.py's tolerances;
and the store's semantics."""
import os
import sys

import numpy as np
import pytest

from test_gicp import FIT_RTOL, T_TOL, make_pair, motion, scene

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
F32 = np.float32
FACE_CELL = 0.25              # the cell size (m) the face cases are laid out for
CELLS_UM = [0, 1, int(FACE_CELL * 1e6), 1_000_000_000]   # automatic, far below / at / far above the spacing


def brute_nn(cloud, q):
    """exact nearest of each query: float32 ((dx*dx)+dy*dy)+dz*dz, lowest index on ties"""
    idx = np.zeros(len(q), np.int32)
    d = np.zeros(len(q), F32)
    for i in range(len(q)):
        dx, dy, dz = (q[i, 0] - cloud[:, 0]), (q[i, 1] - cloud[:, 1]), (q[i, 2] - cloud[:, 2])
        dd = (dx * dx + dy * dy) + dz * dz
        idx[i] = int(np.argmin(dd))
        d[i] = dd[idx[i]]
    return idx, d


def nn_cases():
    """name -> (cloud float32 [n,3], queries float32 [m,3]); every cloud has its bounding-box minimum at
    the origin so that cell faces sit at multiples of the cell size."""
    rng = np.random.default_rng(5)
    cases = {}
    # exact ties between points in different cells: +-0.5 along x and y around queries at cell centres;
    # the tying points are listed in descending cell order, so index order and visit order differ
    c = np.array([[2.125, 2.125, 0.125], [1.125, 3.125, 0.125]], F32)
    off = np.array([[0, 0.5, 0], [0.5, 0, 0], [0, -0.5, 0], [-0.5, 0, 0], [0, 0, 0.5]], F32)
    tie = np.concatenate([ci + off for ci in c] + [np.zeros((1, 3), F32), rng.uniform(0, 4, (200, 3)).astype(F32) + F32(10)])
    cases["ties"] = (tie, c)
    # points exactly on cell faces and +-1 ulp from them, queries on / beside the same faces
    f = np.arange(1, 9, dtype=F32) * F32(FACE_CELL)
    xs = np.concatenate([f, np.nextafter(f, F32(0)), np.nextafter(f, F32(9))])
    face = np.column_stack([xs, np.full_like(xs, F32(0.5)), np.full_like(xs, F32(0.75))])
    face = np.concatenate([np.zeros((1, 3), F32), face, face[:, [1, 0, 2]]])
    fq = np.column_stack([xs + F32(0.01), np.full_like(xs, F32(0.5)), np.full_like(xs, F32(0.75))])
    cases["faces"] = (face, np.concatenate([fq, face[1:40] + F32(0.125), face[1:40]]).astype(F32))
    # duplicate points (the lowest copy wins)
    base = rng.uniform(0, 3, (50, 3)).astype(F32)
    dup = np.concatenate([np.zeros((1, 3), F32), base, base[::-1], base[:10]])
    cases["duplicates"] = (dup, np.concatenate([base[:20], base[:20] + F32(0.01)]))
    # a 10k-point cluster inside one cell of the face grid, plus a sparse surround
    clu = np.concatenate([np.zeros((1, 3), F32), F32(1.0) + rng.uniform(0, 0.2, (10000, 3)).astype(F32),
                          rng.uniform(0, 8, (300, 3)).astype(F32)])
    cases["cluster"] = (clu, np.concatenate([F32(1.0) + rng.uniform(-0.05, 0.25, (60, 3)).astype(F32),
                                             rng.uniform(0, 8, (20, 3)).astype(F32)]))
    # isolated points many shells away from a dense patch, queried from beside them
    iso = np.concatenate([np.zeros((1, 3), F32), rng.uniform(0, 1, (2000, 3)).astype(F32),
                          np.array([[40, 3, 2], [7, 55, 1], [33, 33, 33]], F32)])
    cases["isolated"] = (iso, np.array([[39, 3, 2], [7, 50, 0], [30, 30, 30], [20, 20, 20], [5, 5, 5]], F32))
    # queries far outside the bounding box
    far = np.concatenate([np.zeros((1, 3), F32), rng.uniform(0, 5, (800, 3)).astype(F32)])
    cases["far"] = (far, np.array([[1e5, 2, 2], [-3e4, -3e4, 1], [2, 2, 9e3], [-1e6, 1e6, -1e6], [5.5, 5.5, 5.5]], F32))
    # coordinates around 1e4 and negative (shifted so the minimum stays a face)
    shift = np.array([-10000.0, 10000.0, -9000.0], F32)
    big = np.concatenate([np.zeros((1, 3), F32), rng.uniform(0, 6, (1500, 3)).astype(F32)]) + shift
    cases["large_coords"] = (big, (rng.uniform(-1, 7, (100, 3)).astype(F32) + shift).astype(F32))
    return cases


# ---- CPU: the cases are what they claim to be ------------------------------------------------------------
def test_nn_cases_land_where_intended():
    cases = nn_cases()
    cloud, q = cases["ties"]
    for qi in q:
        d = ((qi[0] - cloud[:, 0]) * (qi[0] - cloud[:, 0]) + (qi[1] - cloud[:, 1]) * (qi[1] - cloud[:, 1])) + \
            (qi[2] - cloud[:, 2]) * (qi[2] - cloud[:, 2])
        hits = np.flatnonzero(d == d.min())
        assert len(hits) >= 5                                              # exact float ties
        cells = [tuple(np.floor(cloud[h, ::-1] / FACE_CELL).astype(int)) for h in hits]   # (z, y, x): key order
        assert len(set(cells)) == len(hits)                                # each in its own cell
        assert hits[0] != hits[min(range(len(hits)), key=lambda i: cells[i])]  # the winner is not visited first
    cloud, q = cases["faces"]
    k = cloud[:, 0] / F32(FACE_CELL)
    assert (k == np.round(k)).sum() >= 8                                   # exactly on faces
    on = np.arange(1, 9, dtype=F32) * F32(FACE_CELL)
    assert np.isin(np.nextafter(on, F32(0)), cloud[:, 0]).all() and np.isin(np.nextafter(on, F32(9)), cloud[:, 0]).all()
    cloud, q = cases["duplicates"]
    idx, d = brute_nn(cloud, q[:20])
    assert (d == 0).all() and (idx <= 50).all()                            # the first copy
    cloud, q = cases["cluster"]
    cl = cloud[1:10001]
    assert (np.floor(cl / FACE_CELL) == np.floor(cl[0] / FACE_CELL)).all()  # one cell
    cloud, q = cases["isolated"]
    idx, d = brute_nn(cloud, q[:3])
    assert list(idx) == [2001, 2002, 2003]
    assert (np.sqrt(brute_nn(cloud[:2001], q[:3])[1]) > 30 * FACE_CELL).all()  # many shells from the patch
    cloud, q = cases["far"]
    assert (np.abs(q[:4]).max(axis=1) > 100 * cloud.max()).all()
    cloud, q = cases["large_coords"]
    shift = cloud[0]
    assert cloud[:, 0].max() < -9990 and cloud[:, 1].min() >= 1e4 and cloud[:, 2].max() < -8990
    for name, (cloud, q) in cases.items():
        assert cloud.dtype == F32 and q.dtype == F32
        lo = shift if name == "large_coords" else 0                          # the box minimum: faces as laid out
        assert (cloud.min(axis=0) == lo).all(), name


def test_bench_gicp_helpers_tiny():
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import bench_gicp
    pts = np.array([[0.1, 0.1, 0.1], [0.2, 0.1, 0.1], [1.1, 0.1, 0.1], [-0.1, 0.0, 0.0]], F32)
    v = bench_gicp.voxel_down(pts, 0.5)
    assert v.dtype == F32 and v.shape == (3, 3)
    assert np.allclose(v[np.argsort(v[:, 0])], [[-0.1, 0, 0], [0.15, 0.1, 0.1], [1.1, 0.1, 0.1]], atol=1e-6)
    w = bench_gicp.make_world(8)
    clouds = bench_gicp.render_clouds(w, w["poses"][:2], 100, leaf=1.0, device="cpu", n_beams=16, n_az=200)
    assert len(clouds) == 2 and all(c.dtype == F32 and c.shape[1] == 3 and len(c) > 50 for c in clouds)
    cands = np.zeros((1, 3), bench_gicp.capi.CAND_DTYPE)
    cands["frame"][0] = [4, -1, 7]
    cands["score"][0] = [3, 9, 5]
    assert list(bench_gicp.visit_order(cands, np.array([3]))[0]) == [1, 2, 0]


# ---- GPU ------------------------------------------------------------------------------------------------
@pytest.fixture
def mgr():
    from sgtd_b200 import capi
    m = capi.STDescManager(device=0)
    yield m
    m.close()


@pytest.mark.gpu
@pytest.mark.parametrize("cell_um", CELLS_UM)
def test_gpu_map_nearest_is_exact(mgr, cell_um):
    mgr.set_option("gicp_cell_um", cell_um)
    cases = nn_cases()
    names = list(cases)
    clouds = [cases[n][0] for n in names]
    off = np.concatenate([[0], np.cumsum([len(c) for c in clouds])]).astype(np.int64)
    mgr.gicp_map_add(np.concatenate(clouds), off, frame_ids=np.arange(100, 100 + len(names)), params=mgr.gicp_params(num_neighbors=1))
    for f, n in enumerate(names):
        cloud, q = cases[n]
        q = np.concatenate([q, cloud[::max(1, len(cloud) // 50)]])            # and queries on stored points
        idx, d = mgr.gicp_map_nearest(100 + f, q)
        ei, ed = brute_nn(cloud, q)
        assert np.array_equal(idx, ei), (n, np.flatnonzero(idx != ei)[:5])
        assert d.tobytes() == ed.tobytes(), n


@pytest.mark.gpu
def test_gpu_map_nearest_device_pointers(mgr):
    import torch
    cloud, q = nn_cases()["cluster"]
    dc = torch.from_numpy(cloud).cuda()
    dq = torch.from_numpy(q).cuda()
    mgr.gicp_map_add(dc.data_ptr(), np.array([0, len(cloud)], np.int64), params=mgr.gicp_params(num_neighbors=5))
    di = torch.zeros(len(q), dtype=torch.int32, device="cuda")
    dd = torch.zeros(len(q), dtype=torch.float32, device="cuda")
    from sgtd_b200 import capi
    mgr._chk(capi.lib().sgtd_gicp_map_nearest(mgr._h, 0, capi._p(dq.data_ptr()), len(q), capi._p(di.data_ptr()), capi._p(dd.data_ptr())))
    ei, ed = brute_nn(cloud, q)
    assert np.array_equal(di.cpu().numpy(), ei) and dd.cpu().numpy().tobytes() == ed.tobytes()


def make_batch(nq, ncand, n_s=500, n_t=1500, seed=0):
    """keyframe clouds (frames 10, 11, ...), query sources seen from near keyframe gt[q] with a known
    motion, and candidates: the right keyframe with a rough loop transform, other keyframes, frame -1 and
    a frame without a stored cloud; one query has no candidate."""
    from sgtd_b200 import capi
    rng = np.random.default_rng(seed)
    nkf = 4
    tgts = [scene(np.random.default_rng(1000 + i), n_t) * F32(1.0 + 0.15 * i) + F32(3 * i) for i in range(nkf)]
    frames = np.arange(10, 10 + nkf)
    srcs, cands, nc, truth = [], np.zeros((nq, ncand), capi.CAND_DTYPE), np.zeros(nq, np.int32), []
    for q in range(nq):
        g = q % nkf
        R, t = motion(rng, 2.0, (0.3, -0.2, 0.04))
        pts = tgts[g][rng.choice(n_t, n_s, replace=False)] + rng.normal(0, 0.01, (n_s, 3))
        srcs.append(((pts - t) @ R).astype(F32))
        truth.append((g, R, t))
        nc[q] = 0 if q % 7 == 3 else ncand
        for c in range(ncand):
            kind = (q + c) % 5
            fr = frames[g] if kind in (0, 3) else (frames[(g + 1) % nkf] if kind == 1 else (-1 if kind == 2 else 99))
            Ri, ti = motion(rng, 1.0, t + rng.normal(0, 0.05, 3))
            cands["frame"][q, c], cands["score"][q, c] = fr, rng.integers(0, 50)
            cands["R"][q, c], cands["t"][q, c] = Ri.reshape(9), ti
    off = np.concatenate([[0], np.cumsum([len(s) for s in srcs])]).astype(np.int64)
    order = np.argsort(-cands["score"], axis=1, kind="stable").astype(np.int32)
    return dict(tgts=tgts, frames=frames, srcs=srcs, src=np.concatenate(srcs), off=off, cands=cands, ncand=nc,
                order=order, truth=truth)


def per_query_loop(mgr, B, prm, use_order):
    by_frame = dict(zip(B["frames"].tolist(), B["tgts"]))
    out = []
    for q, s in enumerate(B["srcs"]):
        n = int(B["ncand"][q])
        c = B["cands"][q, :n]
        targets = [by_frame.get(int(f)) for f in c["frame"]]
        order = B["order"][q, :n] if use_order else None
        if n == 0:
            out.append((-1, np.eye(4)[:3], 100.0, 0))
            continue
        out.append(mgr.gicp_refine_candidates(s, targets, c, order, prm))
    return out


def assert_same(batch, loop):
    chosen, T, fit, nal = batch
    for q, (c, Tq, f, n) in enumerate(loop):
        assert chosen[q] == c and nal[q] == n, (q, chosen[q], c, nal[q], n)
        assert T[q].tobytes() == np.asarray(Tq, np.float64).tobytes() and fit[q] == f, q


@pytest.mark.gpu
@pytest.mark.parametrize("best_fitness", [0.5, 1e-9])
@pytest.mark.parametrize("use_order", [True, False])
@pytest.mark.parametrize("on_device", [False, True])
def test_gpu_refine_batch_is_the_per_query_loop(mgr, best_fitness, use_order, on_device):
    import torch
    B = make_batch(9, 4)
    prm = mgr.gicp_params(max_iterations=10, best_fitness=best_fitness)
    keep = []
    if on_device:
        t = torch.from_numpy(np.concatenate(B["tgts"])).cuda()
        src = torch.from_numpy(B["src"]).cuda()
        keep += [t, src]
        toff = np.concatenate([[0], np.cumsum([len(c) for c in B["tgts"]])]).astype(np.int64)
        mgr.gicp_map_add(t.data_ptr(), toff, frame_ids=B["frames"], params=prm)
        sources = src.data_ptr()
    else:
        for f, c in zip(B["frames"], B["tgts"]):                     # several adds, one cloud each
            mgr.gicp_map_add(c, frame_ids=[f], params=prm)
        sources = B["src"]
    got = mgr.gicp_refine_batch(sources, B["off"], B["cands"], B["ncand"], B["order"] if use_order else None, prm)
    assert_same(got, per_query_loop(mgr, B, prm, use_order))
    assert (got[3] <= B["ncand"]).all() and got[3][3] == 0 and got[0][3] == -1


@pytest.mark.gpu
def test_gpu_refine_batch_wave_size_and_split(mgr):
    """300 queries x 5 candidates of 1,200 source points: with every candidate in one wave the problem
    list needs ~160 MB of scratch and is aligned in two lockstep groups."""
    B = make_batch(300, 5, n_s=1200, seed=3)
    prm = mgr.gicp_params(max_iterations=8, best_fitness=0.5)
    toff = np.concatenate([[0], np.cumsum([len(c) for c in B["tgts"]])]).astype(np.int64)
    mgr.gicp_map_add(np.concatenate(B["tgts"]), toff, frame_ids=B["frames"], params=prm)
    runs = {}
    for w in (0, 1, 3, 1 << 30):
        mgr.set_option("gicp_wave", w)
        runs[w] = mgr.gicp_refine_batch(B["src"], B["off"], B["cands"], B["ncand"], B["order"], prm)
        runs[w] += (mgr.gicp_refine_stats(),)
    for w in (1, 3, 1 << 30):
        for a, b in zip(runs[0][:4], runs[w][:4]):
            assert a.tobytes() == b.tobytes(), w
    problems_all = runs[1 << 30][4][0]
    assert problems_all == int(sum(((B["cands"]["frame"][q, :B["ncand"][q]] >= 0) & (B["cands"]["frame"][q, :B["ncand"][q]] != 99)).sum()
                                   for q in range(300)))
    assert runs[1][4][1] > 1 and runs[1 << 30][4][1] == 1       # waves
    small = dict(B, srcs=B["srcs"][:30], ncand=B["ncand"][:30], cands=B["cands"][:30], order=B["order"][:30])
    assert_same(tuple(a[:30] for a in runs[0][:4]), per_query_loop(mgr, small, prm, True))


@pytest.mark.gpu
def test_gpu_refine_batch_matches_oracle_and_motion(mgr, oracle_lib):
    from sgtd_b200 import capi
    prm = mgr.gicp_params(num_neighbors=20, max_iterations=12, best_fitness=1e-9)
    srcs, tgts, cands, truth = [], [], np.zeros((4, 1), capi.CAND_DTYPE), []
    for i in range(4):
        src, tgt, R, t = make_pair(300 + i, ang=1.5 + i, trans=(0.4, -0.2, 0.03))
        Ri, ti = motion(np.random.default_rng(i), 1.0 + 0.5 * i, (0.35, -0.15, 0.0))
        cands["frame"][i, 0], cands["R"][i, 0], cands["t"][i, 0] = 50 + i, Ri.reshape(9), ti
        srcs.append(src); tgts.append(tgt); truth.append((R, t, Ri, ti))
    toff = np.concatenate([[0], np.cumsum([len(c) for c in tgts])]).astype(np.int64)
    mgr.gicp_map_add(np.concatenate(tgts), toff, frame_ids=50 + np.arange(4), params=prm)
    soff = np.concatenate([[0], np.cumsum([len(c) for c in srcs])]).astype(np.int64)
    chosen, T, fit, nal = mgr.gicp_refine_batch(np.concatenate(srcs), soff, cands, np.ones(4, np.int32), None, prm)
    assert (chosen == 0).all() and (nal == 1).all()
    for i in range(4):
        R, t, Ri, ti = truth[i]
        init = np.column_stack([Ri, ti]).reshape(12)
        Fo, fito, ito, convo = oracle_lib.gicp_align(srcs[i], tgts[i], init12=init, k=20, max_iterations=12)
        assert np.abs(T[i] - Fo[:3]).max() <= T_TOL
        assert abs(fit[i] - fito) <= FIT_RTOL * max(1.0, abs(fito))
        F, fa, it, conv = mgr.gicp_align(srcs[i], tgts[i], init, prm)          # same machinery, with the count
        assert it == ito and conv == convo and F.tobytes() == T[i].tobytes() and fa == fit[i]
        full = np.vstack([T[i], [0, 0, 0, 1]]) @ np.vstack([init.reshape(3, 4), [0, 0, 0, 1]])
        assert np.abs(full[:3, :3] - R).max() < 1e-2 and np.abs(full[:3, 3] - t).max() < 0.1


@pytest.mark.gpu
def test_gpu_store_semantics(mgr):
    from sgtd_b200 import capi
    prm = mgr.gicp_params(num_neighbors=10)
    a, b, c = (scene(np.random.default_rng(s), 400) for s in (1, 2, 3))
    assert mgr.gicp_map_frames() == 0
    mgr.gicp_map_add(np.concatenate([a, b]), [0, 400, 800], params=prm)       # consecutive ids 0, 1
    mgr.gicp_map_add(c, params=prm)                                           # then 2
    assert mgr.gicp_map_frames() == 3
    for f, cl in enumerate((a, b, c)):
        assert np.array_equal(mgr.gicp_map_nearest(f, cl[:30])[0], np.arange(30))
    mgr.gicp_map_add(a, frame_ids=[77], params=prm)
    assert mgr.gicp_map_frames() == 4 and mgr.gicp_map_nearest(77, a[5:6])[0][0] == 5
    for bad in (dict(frame_ids=[2]), dict(frame_ids=[5, 5], offsets=[0, 400, 800])):
        with pytest.raises(capi.SgtdError) as e:
            xyz = np.concatenate([a, b]) if "offsets" in bad else a
            mgr.gicp_map_add(xyz, bad.get("offsets"), frame_ids=bad["frame_ids"], params=prm)
        assert e.value.status == capi.E_INVALID
    with pytest.raises(capi.SgtdError) as e:                                  # num_neighbors differs
        mgr.gicp_map_add(b, frame_ids=[90], params=mgr.gicp_params(num_neighbors=12))
    assert e.value.status == capi.E_INVALID
    with pytest.raises(capi.SgtdError) as e:                                  # cloud smaller than k
        mgr.gicp_map_add(a[:9], frame_ids=[91], params=prm)
    assert e.value.status == capi.E_INVALID
    cand = np.zeros((1, 1), capi.CAND_DTYPE)
    cand["R"][0, 0] = np.eye(3).reshape(9)
    with pytest.raises(capi.SgtdError) as e:                                  # source smaller than k
        mgr.gicp_refine_batch(a[:9], [0, 9], cand, [1], None, prm)
    assert e.value.status == capi.E_INVALID
    with pytest.raises(capi.SgtdError) as e:
        mgr.gicp_map_nearest(5, a[:3])
    assert e.value.status == capi.E_INVALID
    assert mgr.gicp_map_frames() == 4
    mgr.gicp_map_clear()
    assert mgr.gicp_map_frames() == 0
    chosen, T, fit, nal = mgr.gicp_refine_batch(a, [0, 400], cand, [1], None, prm)   # nothing stored: skipped
    assert chosen[0] == -1 and nal[0] == 0 and fit[0] == 100.0
    mgr.gicp_map_add(c, params=mgr.gicp_params(num_neighbors=12))             # re-add, any k after a clear
    assert mgr.gicp_map_frames() == 1 and mgr.gicp_map_nearest(0, c[:4])[0].tolist() == [0, 1, 2, 3]
