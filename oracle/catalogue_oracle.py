"""numpy / Python restatement of the integer-coded part of preprocess.py:main() (:269-375), independent of the CUDA
path (pert_gnn_kdd23_b200/catalogue.py).  Patterns are compared as tuples of (um, dm, interface) triples, which is
what joining the integer ids with "_" and " " (:280-289) compares.

-> dict of numpy arrays in the layout of ``catalogue.Catalogue``:
  traceid, entry, runtime_id, timestamp, y          per trace, tr2data order (entry asc, traceid asc)
  pat_runtime_id, pat_traceid, pat_occurrences      per pattern, runtime2graph insertion order
  entries, ent_ptr, ent_runtime_id, ent_prob        entry2runtimes as a CSR (float64 probabilities)
"""
import numpy as np


def catalogue(table):
    tid = np.asarray(table["traceid"], dtype=np.int64)
    order = np.argsort(tid, kind="stable")                         # groupby("traceid"): file order inside a trace
    traceids, starts = np.unique(tid[order], return_index=True)
    ends = np.append(starts[1:], len(order))
    um, dm, itf = (np.asarray(table[c], dtype=np.int64) for c in ("um", "dm", "interface"))
    rt, ts, ent = (np.asarray(table[c], dtype=np.int64) for c in ("rt", "timestamp", "entryid"))
    T = len(traceids)
    rid, entry, bucket, y = (np.empty(T, dtype=np.int64) for _ in range(4))
    ids = {}
    for t in range(T):
        rows = order[starts[t]:ends[t]]
        seq = tuple(zip(um[rows].tolist(), dm[rows].tolist(), itf[rows].tolist()))
        rid[t] = ids.setdefault(seq, len(ids))                     # factorize: first appearance, traceid order
        e = np.unique(ent[rows])
        if len(e) != 1:
            raise ValueError(f"trace {traceids[t]} has entryids {e.tolist()}")
        entry[t] = e[0]
        bucket[t] = ts[rows].min() // 30000 * 30000                # :39
        y[t] = np.abs(rt[rows]).max()                              # :290-292
    eorder = np.argsort(entry, kind="stable")                      # groupby("entryid") then groupby("traceid")
    counts, rep, occ = {}, {}, {}
    for t in eorder.tolist():
        e, r = int(entry[t]), int(rid[t])
        c = counts.setdefault(e, {})
        c[r] = c.get(r, 0) + 1
        rep.setdefault(r, t)
        occ[r] = occ.get(r, 0) + 1
    entries = sorted(counts)
    ent_ptr, ent_rid, ent_prob = [0], [], []
    for e in entries:
        total = sum(counts[e].values())
        for r, n in counts[e].items():
            ent_rid.append(r)
            ent_prob.append(n / total)                             # :371-375
        ent_ptr.append(len(ent_rid))
    pats = list(rep)
    return {"traceid": traceids[eorder], "entry": entry[eorder], "runtime_id": rid[eorder],
            "timestamp": bucket[eorder], "y": y[eorder],
            "pat_runtime_id": np.array(pats, dtype=np.int64),
            "pat_traceid": traceids[np.array([rep[r] for r in pats], dtype=np.int64)],
            "pat_occurrences": np.array([occ[r] for r in pats], dtype=np.int64),
            "entries": np.array(entries, dtype=np.int64), "ent_ptr": np.array(ent_ptr, dtype=np.int64),
            "ent_runtime_id": np.array(ent_rid, dtype=np.int64), "ent_prob": np.array(ent_prob, dtype=np.float64)}


def representative_rows(table, traceids):
    """Raw rows (file order) of each given trace -> (dict of int64 columns, row_ptr)."""
    tid = np.asarray(table["traceid"], dtype=np.int64)
    idx = [np.flatnonzero(tid == t) for t in np.asarray(traceids).tolist()]
    row_ptr = np.concatenate([[0], np.cumsum([len(i) for i in idx])]).astype(np.int64)
    rows = np.concatenate(idx)
    return {k: np.asarray(v, dtype=np.int64)[rows] for k, v in table.items()}, row_ptr
