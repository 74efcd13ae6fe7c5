"""Shape of the first pass's containment resolution for a bench.py workload, on the CPU (exact, no GPU needed).

    python profiles/resolve_shape.py [--workload c3] [--out FILE]

Events are the oracle's per-record types on the workload's flat piles: KB = victim a, container b; KA = victim b,
container a; time = record index.  The earliest-event test of k_resolve_fast (containment.cu) settles victim v at its
earliest event (t1, c1) when c1 == v, c1 has no event, or c1's earliest event is later than t1; the others are "hard".
The script checks those death times against a sequential pass, counts what is left to k_resolve (hard victims, their
events, the events the filter drops because their container is settled to die first), and the depth of the dependencies:
settled victims per round of a one-event-per-round Jacobi sweep.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

INF = np.iinfo(np.int64).max


def events(ds, piles):
    from oracle import oracle as O
    rec = np.ascontiguousarray(ds.records, dtype=np.uint32).reshape(-1, 7)
    _, ty = O.trim_type_batch(rec, piles)
    valid = (rec[:, 6] & 2) == 0
    a, b = rec[:, 0].astype(np.int64), rec[:, 1].astype(np.int64)
    isb, isa = (ty == O.KB) & valid, (ty == O.KA) & valid
    t = np.flatnonzero(isa | isb)
    return np.where(isb[t], a[t], b[t]), np.where(isb[t], b[t], a[t]), t.astype(np.int64), int(rec.shape[0])


def sequential(v, c, t, n):
    alive = np.ones(n, bool)
    D = np.full(n, INF)
    for vv, cc, tt in zip(v.tolist(), c.tolist(), t.tolist()):   # t ascending
        if alive[vv] and alive[cc]:
            alive[vv] = False
            D[vv] = tt
    return D


def jacobi_rounds(vs, cs, ts, first, n, D_want):
    """Every open victim looks at its earliest event not known to be void: it fires when the container is the victim,
    is settled to die later, or is open with a later lower bound; it is void when the container is settled to die earlier
    (the pointer moves on, the victim stays open).  Settled victims per round until none is open."""
    vid = vs[first]
    end = np.r_[first[1:], vs.size]
    ptr = first.copy()
    D = np.full(n, INF)
    settled = np.ones(n, bool)
    settled[vid] = False
    lb = np.full(n, INF)                  # lower bound of an open victim: time of its current event
    lb[vid] = ts[first]
    open_ = np.arange(vid.size)
    per_round = []
    while open_.size:
        p = ptr[open_]
        v = vid[open_]
        done = p >= end[open_]
        q = np.minimum(p, vs.size - 1)
        c, t = cs[q], ts[q]
        c_set = settled[c]
        fire = ~done & ((c == v) | (c_set & (D[c] > t)) | (~c_set & (lb[c] > t)))
        void = ~done & ~fire & c_set
        fin = done | fire
        D[v[fire]] = t[fire]
        settled[v[fin]] = True
        ptr[open_[void]] += 1
        nv = open_[void]
        lb[vid[nv]] = np.where(ptr[nv] < end[nv], ts[np.minimum(ptr[nv], vs.size - 1)], INF)
        per_round.append(int(fin.sum()))
        open_ = open_[~fin]
    assert np.array_equal(D[vid], D_want[vid]), "Jacobi sweep differs from the sequential pass"
    return per_round


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="c3")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import bench
    t0 = time.time()
    ds = bench.make_dataset(args.workload, 1)
    piles = ds.flat_piles()
    n = piles.shape[0]
    v, c, t, n_rec = events(ds, piles)
    D = sequential(v, c, t, n)
    o = np.lexsort((t, v))
    vs, cs, ts = v[o], c[o], t[o]
    first = np.r_[0, np.flatnonzero(np.diff(vs)) + 1] if vs.size else np.zeros(0, np.int64)
    fv, fc, ft = vs[first], cs[first], ts[first]
    tmin = np.full(n, INF)
    tmin[fv] = ft
    easy = (fc == fv) | (tmin[fc] > ft)
    easy_ok = bool(np.array_equal(D[fv[easy]], ft[easy]))
    S_easy = np.full(n, -1)               # death time of the piles the test settled; -1 = not settled by it
    S_easy[fv[easy]] = ft[easy]
    hard = np.zeros(n, bool)
    hard[fv[~easy]] = True
    ev_hard = hard[v]
    dropped = ev_hard & (S_easy[c] >= 0) & (S_easy[c] < t)   # container settled to die before the event: void
    rounds = jacobi_rounds(vs, cs, ts, first, n, D)
    out = {"workload": bench.WORKLOADS[args.workload][3], "records": n_rec, "piles": int(n), "events": int(t.size),
           "victims": int(fv.size), "dying": int(np.sum(D != INF)),
           "easy": int(easy.sum()), "easy_death_times_match_sequential": easy_ok,
           "easy_by_branch": {"self": int(np.sum(fc == fv)), "container_without_events": int(np.sum((fc != fv) & (tmin[fc] == INF))),
                              "container_first_event_later": int(np.sum((fc != fv) & (tmin[fc] != INF) & (tmin[fc] > ft)))},
           "hard": int((~easy).sum()), "events_of_hard": int(ev_hard.sum()),
           "events_of_hard_dropped_as_void": int(dropped.sum()), "events_of_hard_kept": int((ev_hard & ~dropped).sum()),
           "jacobi_rounds": len(rounds), "jacobi_settled_per_round": rounds,
           "seconds": round(time.time() - t0, 1)}
    text = json.dumps(out, indent=1)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text + "\n")
    print(text)


if __name__ == "__main__":
    main()
