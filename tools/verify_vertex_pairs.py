"""How many distinct (query vertex, DB vertex) pairs the verification of a candidate tests.

candidate_verify's vertex test depends on one query vertex, one DB vertex and the hypothesis only, so k_verify
(sgtd_b200/csrc/search.cu) tests each distinct pair once per hypothesis instead of the three vertices of every
match.  This script counts, with the CPU oracle on the bench's own generator (synth.make_config), per candidate:
matches M, vertex tests 3M, distinct pairs U (keyed by the bits of the six coordinates, as the kernel keys them),
distinct query / DB vertices, and the chunks k_verify takes at its default table size.

    python tools/verify_vertex_pairs.py                                  # configs[3], 3,000 keyframes, 12 queries
    python tools/verify_vertex_pairs.py --keyframes 100000 --queries 1024 --sample 16   # the bench workload

--sample n takes n queries spread evenly over the batch (the oracle searches a 100k-keyframe DB at a few
queries per second).
"""
import argparse
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from oracle import orc  # noqa: E402
from sgtd_b200 import synth  # noqa: E402

PAIR_CAP, CHUNK_MATCHES = 768, 2048  # k_verify: kPairCap, kChunkMatches


def chunks(qv, dv, M, cap=PAIR_CAP, chunk_matches=CHUNK_MATCHES):
    """chunks k_verify takes: a chunk ends at the first match whose new pairs do not fit the table, or after
    chunk_matches matches, and the next one starts with an empty table.  Holes (ids reserved by racing inserts
    of the same pair) can end a chunk earlier on the GPU; this counts none."""
    keys = np.concatenate([qv, dv], 1).reshape(M, 3, 6)
    n, j = 0, 0
    while j < M:
        n += 1
        seen, cb = set(), j
        while j < M and j - cb < chunk_matches:
            new = {k.tobytes() for k in keys[j]} - seen
            if len(seen) + len(new) > cap:
                break
            seen |= new
            j += 1
    return n


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--config", type=int, default=3)
    ap.add_argument("--keyframes", type=int, default=3000)
    ap.add_argument("--queries", type=int, default=12)
    ap.add_argument("--sample", type=int, default=0, help="queries to search, spread over the batch (0 = all)")
    ap.add_argument("--threads", type=int, default=os.cpu_count())
    a = ap.parse_args()
    t0 = time.time()
    cfg = synth.make_config(a.config, a.keyframes, a.queries)
    xyz, lab, off = cfg["db"]
    qx, ql, qo = cfg["queries"]
    o = orc.Oracle()
    o.build_add_many(xyz, lab, off, nthreads=a.threads)
    # DB descriptors by global index, for the keyframes the candidates name (same arithmetic as the DB build)
    nf = len(off) - 1
    start = np.zeros(nf + 1, np.int64)
    per = {}
    o2 = orc.Oracle()

    def frame_descs(f):
        if f not in per:
            try:
                per[f] = o2.build(xyz[off[f]:off[f + 1]], lab[off[f]:off[f + 1]])
            except ValueError:
                per[f] = np.zeros(0, orc.DESC_DTYPE)
        return per[f]

    for f in range(nf):
        start[f + 1] = start[f] + len(frame_descs(f))
        if a.keyframes > 20000:
            per.pop(f)
    nq = len(qo) - 1
    qs = range(nq) if a.sample <= 0 else sorted(set(np.linspace(0, nq - 1, a.sample).astype(int).tolist()))
    rows = []
    for i in qs:
        q = o2.build(qx[qo[i]:qo[i + 1]], ql[qo[i]:qo[i + 1]])
        r = o.search(q, nthreads=a.threads, want_votes=False)
        mo = 0
        for c in r["cands"]:
            M = int(c["nmatch"])
            mq, mg = r["m_q"][mo:mo + M], r["m_g"][mo:mo + M].astype(np.int64)
            mo += M
            if M == 0:
                continue
            f = int(c["frame"])
            d = frame_descs(f)
            assert len(d) == start[f + 1] - start[f] and ((mg >= start[f]) & (mg < start[f + 1])).all()
            qv = q["vert"][mq].reshape(M, 3, 3).view(np.uint32).reshape(M * 3, 3)
            dv = d["vert"][mg - start[f]].reshape(M, 3, 3).view(np.uint32).reshape(M * 3, 3)
            U = np.unique(np.concatenate([qv, dv], 1), axis=0).shape[0]
            rows.append((M, U, np.unique(qv, axis=0).shape[0], np.unique(dv, axis=0).shape[0],
                         chunks(qv, dv, M)))
    rows = np.array(rows, np.int64).reshape(-1, 5)
    M, U, Uq, Ud, nch = rows.T
    print("config %d, %d keyframes, %d of %d queries, %d candidates with matches (%.0f s)"
          % (a.config, a.keyframes, len(qs), nq, len(rows), time.time() - t0))
    print("| per candidate | median | max |")
    print("|---|---|---|")
    for name, v in (("matches M", M), ("vertex tests 3M", 3 * M), ("distinct (query vertex, DB vertex) pairs U", U),
                    ("distinct query vertices", Uq), ("distinct DB vertices", Ud), ("k_verify chunks", nch)):
        print("| %s | %g | %d |" % (name, np.median(v), v.max()))
    print("sum U / sum 3M = %.4f; candidates in one chunk: %.4f" % (U.sum() / (3 * M.sum()), (nch == 1).mean()))


if __name__ == "__main__":
    main()
