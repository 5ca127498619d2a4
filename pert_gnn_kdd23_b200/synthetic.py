"""Seeded synthetic call-graph generator for the BASELINE.json configurations.

The reference trains on the Alibaba 2021 micro-service traces (200 GB, not
available); its per-sample tensor schema is reference pert_gnn.py:163-173.
This module emits ``Data`` objects of exactly that schema with the shapes
SURVEY.md section 8d defines:

  x [n,9] f32 (8 resource stats + missing indicator, stats zeroed where the
  indicator is 1 -- mirrors pert_gnn.py:44-66), edge_index [2,e] i64,
  edge_attr [e,2|4] i64 (interface id, rpctype id[, call_ind, same_ms]),
  cat_X [n,1] i64 (micro-service id), node_depth [n,1] i64,
  pattern_num_nodes [n,1] f32, pattern_probs [P,1] f32, entry_id [1] i64,
  y 0-dim i64, plus ``rt_probs`` [n,1] f32 = the per-node pattern probability the
  reference's train loop rebuilds on the host every step (pert_gnn.py:220-230).

DAG law: n nodes on L levels, node 0 the sole root (level 0); every other node
gets one parent drawn uniformly from the previous level (so every node is reachable);
the remaining m-(n-1) edges are uniform (lower level -> strictly higher level)
pairs, no duplicates; node ids (except the root) and the edge order are
shuffled -- sorting is part of the measured collation.
"""
from __future__ import annotations

import math

import numpy as np
import torch

from .data import Data

N_MS, N_IF, N_RPC, N_ENTRY, N_FEAT = 4096, 1024, 8, 64, 9

# id -> (graphs, nodes, edges, hidden, num_layers, levels);  nodes=None => power law
CONFIGS = {
    1: dict(graphs=64, nodes=50, edges=150, hidden=32, num_layers=1, levels=5),
    2: dict(graphs=256, nodes=200, edges=600, hidden=64, num_layers=3, levels=8),
    3: dict(graphs=1024, nodes=None, edges=None, hidden=128, num_layers=3, levels=None),
    4: dict(graphs=4096, nodes=200, edges=600, hidden=128, num_layers=3, levels=8),
    5: dict(graphs=256, nodes=1000, edges=3000, hidden=128, num_layers=5, levels=12),
}


def model_args(cfg_id):
    """Positional ctor args of SAGEDeterministic for a config (SURVEY.md 8d)."""
    c = CONFIGS[cfg_id]
    return (N_FEAT, [N_MS], N_ENTRY - 1, N_IF - 1, N_RPC - 1, c["hidden"], c["num_layers"], 0.0)


def _level_sizes(rng, n, L):
    L = max(1, min(L, n))
    if L == 1:
        return np.array([n], dtype=np.int64)
    sizes = np.ones(L, dtype=np.int64)
    extra = n - L
    if extra > 0:
        sizes[1:] += np.bincount(rng.integers(1, L, size=extra), minlength=L)[1:] if L > 1 else 0
    return sizes


def random_dag(rng, n, m, L):
    """Returns (edge_index int64 [2,m'], level int64 [n]); m' = min(m, max possible)."""
    sizes = _level_sizes(rng, n, L)
    L = len(sizes)
    level_sorted = np.repeat(np.arange(L), sizes)               # level of position p (sorted)
    ids = np.concatenate([[0], 1 + rng.permutation(n - 1)]) if n > 1 else np.array([0])
    level = np.empty(n, dtype=np.int64)
    level[ids] = level_sorted
    starts = np.concatenate([[0], np.cumsum(sizes)])
    # spanning tree: parent uniform in previous level
    pos = np.arange(sizes[0], n)
    lv = level_sorted[pos]
    par_pos = starts[lv - 1] + (rng.random(pos.shape[0]) * sizes[lv - 1]).astype(np.int64)
    src = ids[par_pos]
    dst = ids[pos]
    have = set((src * n + dst).tolist())
    # cap by the number of admissible (lower -> strictly higher level) pairs
    cum = np.cumsum(sizes)
    max_pairs = int(sum(int(sizes[l]) * int(n - cum[l]) for l in range(L)))
    m = min(m, max_pairs)
    extra_s, extra_d = [], []
    need = m - (n - 1)
    while need > 0:
        k = max(64, 3 * need)
        u = rng.integers(0, n, size=k)
        v = rng.integers(0, n, size=k)
        ok = level[u] < level[v]
        for a, b in zip(u[ok].tolist(), v[ok].tolist()):
            key = a * n + b
            if key not in have:
                have.add(key)
                extra_s.append(a)
                extra_d.append(b)
                need -= 1
                if need == 0:
                    break
    src = np.concatenate([src, np.array(extra_s, dtype=np.int64)])
    dst = np.concatenate([dst, np.array(extra_d, dtype=np.int64)])
    order = rng.permutation(src.shape[0])
    return np.stack([src[order], dst[order]]).astype(np.int64), level


def bfs_min_depth(edge_index, n, root=0):
    """Min hop depth from ``root`` over out-edges (what misc.py:59-63 computes); -1 if unreachable."""
    depth = np.full(n, -1, dtype=np.int64)
    depth[root] = 0
    src, dst = edge_index
    frontier = np.zeros(n, dtype=bool)
    frontier[root] = True
    d = 0
    while frontier.any():
        nxt = np.zeros(n, dtype=bool)
        nxt[dst[frontier[src]]] = True
        nxt &= depth < 0
        d += 1
        depth[nxt] = d
        frontier = nxt
    return depth


def _node_depth(depth):
    # reference quirk (misc.py:159-175,215): unreachable -> 0, depth/max truncated to long -> {0,1}
    d = np.where(depth < 0, 0, depth).astype(np.float64)
    mx = d.max() if d.max() > 0 else 1.0
    return (d / mx).astype(np.int64).reshape(-1, 1)


def make_graph(rng, n, m, L, patterns=1, edge_attr_cols=2):
    """One reference-schema ``Data``: disjoint union of ``patterns`` runtime-pattern
    DAGs (pert_gnn.py:134-173)."""
    eis, levels, depths, pnn, rtp = [], [], [], [], []
    probs = rng.random(patterns) + 0.1
    probs = probs / probs.sum()
    off = 0
    for p in range(patterns):
        np_ = n if patterns == 1 else max(2, int(n // patterns))
        mp_ = m if patterns == 1 else max(np_ - 1, int(m // patterns))
        ei, lv = random_dag(rng, np_, mp_, L)
        eis.append(ei + off)
        levels.append(lv)
        depths.append(bfs_min_depth(ei, np_, 0))
        pnn.append(np.full((np_, 1), float(np_), dtype=np.float32))
        rtp.append(np.full((np_, 1), float(probs[p]), dtype=np.float32))
        off += np_
    edge_index = np.concatenate(eis, axis=1)
    level = np.concatenate(levels)
    nn_, ne = off, edge_index.shape[1]
    x = rng.random((nn_, N_FEAT), dtype=np.float32)
    miss = rng.random(nn_) < 0.2
    x[:, 8] = miss.astype(np.float32)
    x[miss, :8] = 0.0
    ea = np.zeros((ne, edge_attr_cols), dtype=np.int64)
    ea[:, 0] = rng.integers(0, N_IF, size=ne)
    ea[:, 1] = rng.integers(0, N_RPC, size=ne)
    if edge_attr_cols == 4:
        ea[:, 2] = rng.integers(0, 2, size=ne)
        ea[:, 3] = rng.integers(0, 2, size=ne)
    return Data(
        x=torch.from_numpy(x),
        edge_index=torch.from_numpy(edge_index),
        edge_attr=torch.from_numpy(ea),
        cat_X=torch.from_numpy(rng.integers(0, N_MS, size=(nn_, 1))),
        node_depth=torch.from_numpy(np.concatenate([_node_depth(d) for d in depths])),
        pattern_num_nodes=torch.from_numpy(np.concatenate(pnn)),
        pattern_probs=torch.from_numpy(probs.astype(np.float32).reshape(-1, 1)),
        entry_id=torch.from_numpy(rng.integers(0, N_ENTRY, size=1)),
        y=torch.tensor(int(rng.integers(1, 5000)), dtype=torch.long),
        rt_probs=torch.from_numpy(np.concatenate(rtp)),
        level=torch.from_numpy(level),
        min_depth=torch.from_numpy(np.concatenate(depths)),
    )


def _powerlaw_nodes(rng, lo=20, hi=500, alpha=1.5):
    # truncated Pareto(alpha) on [lo, hi] by inverse CDF
    u = rng.random()
    a = lo ** (-alpha)
    b = hi ** (-alpha)
    return int((a - u * (a - b)) ** (-1.0 / alpha))


def make_data_list(cfg_id, num_graphs=None, seed=None, patterns=1, edge_attr_cols=2, jitter=0.0):
    """List of ``Data`` for one BASELINE config; seed defaults to 1000+cfg_id.  ``jitter`` j draws every graph's node
    count uniformly from nodes*(1 +- j) (edges scale with it): BASELINE says "~200 nodes / ~600 edges"."""
    c = CONFIGS[cfg_id]
    rng = np.random.default_rng(1000 + cfg_id if seed is None else seed)
    out = []
    for _ in range(c["graphs"] if num_graphs is None else num_graphs):
        if c["nodes"] is None:
            n = _powerlaw_nodes(rng)
            m = 3 * n
            L = int(min(10, max(3, round(math.log2(n)))))
        else:
            n, m, L = c["nodes"], c["edges"], c["levels"]
            if jitter > 0:
                n = max(2, int(round(n * (1.0 + jitter * (2.0 * rng.random() - 1.0)))))
                m = int(round(n * c["edges"] / c["nodes"]))
        out.append(make_graph(rng, n, m, L, patterns=patterns, edge_attr_cols=edge_attr_cols))
    return out


# ------------------------------------------------------------------------------------------------------------------
# Synthetic "processed/" artefacts in the reference's own schema (what preprocess.py:378-381 writes and pert_gnn.py:
# 297-305 loads): the inputs of get_entry_data / get_data_list (pert_gnn.py:134-188).  Used to run the reference's
# own sample assembly + train/test loop (oracle/gen_golden_loop.py -> tests/golden/ref_loop.npz) and, with the same
# seed, the device-side pattern store (store.py).
def make_trace_artifacts(seed=7, n_ms=48, n_patterns=14, n_entries=6, n_traces=72, n_timestamps=5, n_if=32, n_rpc=6,
                         nodes=(5, 40), resource_frac=0.7, y_max=10, runtime2graph=None, patterns_per_entry=(1, 3)):
    """-> dict(runtime2graph, entry2runtimes, tr2data, resource_index [(timestamp, msname)], resource_values [R,8],
    n_ms, n_if, n_rpc).
      runtime2graph[rt] = {edge_index [2,e] i64, edge_attr [e,4] i64, ms_id [n,1] i64, num_nodes int, node_depth [n,1] i64}
      entry2runtimes[entry] = {rt: prob}        (probabilities of an entry's runtime patterns sum to 1)
      tr2data[trace] = {entry_id int, timestamp int, y 0-dim i64 tensor}
    Microservice ids repeat inside a pattern (PERT graphs have several stage nodes per microservice), which exercises
    the last-occurrence rule of the reference's feature join (pert_gnn.py:54-65)."""
    rng = np.random.default_rng(seed)
    given = runtime2graph is not None          # patterns built elsewhere (e.g. pertgraph.build_pert_graphs)
    runtime2graph = dict(runtime2graph) if given else {}
    for rt in range(0 if given else n_patterns):
        n = int(rng.integers(nodes[0], nodes[1] + 1))
        m = min(3 * n, n * (n - 1) // 2)
        L = int(min(6, max(2, round(math.log2(n)))))
        ei, _ = random_dag(rng, n, m, L)
        e = ei.shape[1]
        ea = np.stack([rng.integers(0, n_if, e), rng.integers(0, n_rpc, e), rng.integers(0, 2, e),
                       rng.integers(0, 2, e)], axis=1).astype(np.int64)
        ms = rng.integers(0, n_ms, size=(n, 1)).astype(np.int64)
        if n >= 4:
            ms[n - 1, 0] = ms[0, 0]                     # guaranteed duplicate microservice inside the pattern
        runtime2graph[100 + rt] = {
            "edge_index": torch.from_numpy(ei), "edge_attr": torch.from_numpy(ea), "ms_id": torch.from_numpy(ms),
            "num_nodes": n, "node_depth": torch.from_numpy(_node_depth(bfs_min_depth(ei, n, 0))),
        }
    rts = list(runtime2graph.keys())
    entry2runtimes = {}
    for entry in range(n_entries):
        k = int(rng.integers(patterns_per_entry[0], patterns_per_entry[1] + 1))
        chosen = [int(x) for x in rng.choice(rts, size=k, replace=False)]
        p = rng.random(k) + 0.2
        p = p / p.sum()
        entry2runtimes[entry] = {rt: float(pp) for rt, pp in zip(chosen, p)}
    timestamps = [int(60000 * (t + 1)) for t in range(n_timestamps)]
    tr2data = {}
    for tr in range(n_traces):
        tr2data[f"trace{tr:04d}"] = {"entry_id": int(rng.integers(0, n_entries)),
                                     "timestamp": int(timestamps[int(rng.integers(0, n_timestamps))]),
                                     "y": torch.tensor(int(rng.integers(1, y_max)))}
    with_res = np.sort(rng.choice(n_ms, size=max(1, int(resource_frac * n_ms)), replace=False))
    index = [(t, int(ms)) for t in timestamps for ms in with_res]       # every resourced ms has every timestamp
    values = rng.random((len(index), N_FEAT - 1)).astype(np.float64)     # read back from CSV as float64
    return {"runtime2graph": runtime2graph, "entry2runtimes": entry2runtimes, "tr2data": tr2data,
            "resource_index": index, "resource_values": values, "n_ms": n_ms, "n_if": n_if, "n_rpc": n_rpc}


def make_span_tables(seed=11, n_traces=24, n_ms=40, calls=(1, 30), n_if=32, n_rpc=6, anomalies=True):
    """Raw per-trace span tables with the columns the reference's preprocessing hands to GraphConstruct
    (preprocess.py:296-318: timestamp, rpcid, um, rpctype, dm, interface, rt, endTimestamp = timestamp + |rt|, :263),
    all int64.  -> list of dicts.  The first generated call (root -> entry service) has the strictly largest |rt| and
    the smallest timestamp, which is how misc.py:138-142 identifies the root.  Timestamps are coarse on purpose
    (many ties, zero-length calls) and, with ``anomalies``, the rows include what misc.py:87-105 drop_wrong_edges
    removes: self loops, repeated rpcids, calls back to the root, repeated (um, dm) pairs and reversed pairs."""
    rng = np.random.default_rng(seed)
    out = []
    for _ in range(n_traces):
        m = int(rng.integers(calls[0], calls[1] + 1))
        root, entry = (int(v) for v in rng.choice(n_ms, size=2, replace=False))
        t0 = int(rng.integers(1000, 5000))
        rows = [[t0, root, entry, 200 + int(rng.integers(0, 50))]]     # timestamp, um, dm, rt
        called = [entry]
        for _k in range(m - 1):
            um = called[int(rng.integers(0, len(called)))] if rng.random() < 0.8 else int(rng.integers(0, n_ms))
            dm = int(rng.integers(0, n_ms))
            if anomalies and rng.random() < 0.06:
                dm = um                                              # self loop
            elif anomalies and rng.random() < 0.06:
                dm = root                                            # call back to the root
            elif anomalies and rng.random() < 0.08 and len(rows) > 1:
                o = rows[int(rng.integers(1, len(rows)))]
                um, dm = (o[1], o[2]) if rng.random() < 0.5 else (o[2], o[1])   # repeated / reversed pair
            rt = int(rng.integers(0, 6)) * (1 if rng.random() < 0.5 else -1)
            rows.append([t0 + int(rng.integers(0, 8)), um, dm, rt])
            called.append(dm)
        rows = np.array(rows, dtype=np.int64)
        rows = rows[rng.permutation(len(rows))]
        n = len(rows)
        rpcid = np.arange(n, dtype=np.int64)
        if anomalies and n > 3:
            for _d in range(int(rng.integers(0, 3))):
                a, b = rng.integers(0, n, size=2)
                rpcid[a] = rpcid[b]                                  # repeated rpcid
        out.append({"timestamp": rows[:, 0].copy(), "um": rows[:, 1].copy(), "dm": rows[:, 2].copy(),
                    "rt": rows[:, 3].copy(), "rpcid": rpcid, "interface": rng.integers(0, n_if, n).astype(np.int64),
                    "rpctype": rng.integers(0, n_rpc, n).astype(np.int64),
                    "endTimestamp": rows[:, 0] + np.abs(rows[:, 3])})
    return out


def make_pert_artifacts(seed=3, n_patterns=256, n_entries=64, n_traces=4096, calls=(60, 72), device="cuda", n_ms=4096,
                        n_if=1024, n_rpc=8, kind="pert"):
    """PERT-exact synthetic artefacts (SURVEY N2): span tables -> host row filters (misc.py:87-105,138-142) -> PERT (or
    span) graphs built ON THE GPU (pertgraph.build_pert_graphs) -> the processed/ artefact schema of
    make_trace_artifacts with ONE pattern per entry, so a trace's sample is one PERT graph (nodes = 2 calls + distinct
    microservices, edges = 4 calls).  -> (artifacts, info) with info = rows / nodes / edges / seconds of the build."""
    import time

    from . import pertgraph

    tabs = make_span_tables(seed, n_patterns, n_ms=n_ms, calls=calls, n_if=n_if, n_rpc=n_rpc, anomalies=False)
    tables, roots = [], []
    for tab in tabs:
        root = pertgraph.get_root_ms(tab)
        keep = pertgraph.drop_wrong_edges(tab, root)
        tables.append({k: v[keep] for k, v in tab.items()})
        roots.append(root)
    torch.cuda.synchronize(device)
    t0 = time.perf_counter()
    pg = pertgraph.build_pert_graphs(tables, roots, device, kind=kind).check()
    torch.cuda.synchronize(device)
    secs = time.perf_counter() - t0
    # entries / traces / resources around the patterns; the pattern dict only carries the ids here (the graphs stay on the
    # device: art["graphs"] + art["runtime_ids"] go to PatternStore.from_graphs)
    ids = [100 + i for i in range(len(pg))]
    art = make_trace_artifacts(seed, n_ms=n_ms, n_entries=n_entries, n_traces=n_traces, n_if=n_if, n_rpc=n_rpc,
                               y_max=5000, runtime2graph={i: None for i in ids}, patterns_per_entry=(1, 1))
    art["graphs"], art["runtime_ids"] = pg, ids
    info = {"patterns": len(pg), "span_rows": int(sum(len(t["um"]) for t in tables)), "nodes": int(pg.node_ptr[-1]),
            "edges": int(pg.edge_ptr[-1]), "build_s": secs}
    return art, info


RESOURCE_COLUMNS = tuple(f"instance_{k}_usage_{s}" for k in ("cpu", "memory") for s in ("max", "min", "mean", "median"))


def make_processed_tables(seed=5, n_traces=300, n_patterns=24, n_entries=8, n_ms=30, rows=(1, 12), n_if=16, n_rpc=4,
                          traceid_base=0):
    """Seeded span table in the ``processed/processed_df.csv`` schema (what preprocess.py:main() reads; int64 columns
    traceid, timestamp, rpcid, um, dm, interface, rpctype, rt, entryid) + the matching ``processed_resource_df.csv``
    (timestamp, msname, 8 statistics) with a row for every (30 s bucket of a trace, microservice), as main() needs.
    -> (table: dict of int64 arrays in file order, resource: dict of arrays).

    Patterns are (um, dm, interface) sequences; the traces of one pattern differ in rpctype, rpcid, timestamps and rt.
    Row 0 of every pattern is the root call (the largest |rt| at the smallest timestamp; its um occurs nowhere else).
    The table has self loops and repeated rpcids, one pattern under two entries, single-row traces, traces starting
    next to a 30 s bucket boundary, non-dense traceids (+ ``traceid_base``) and entry ids with gaps; rows are sorted by
    timestamp (as get_df leaves them), so traces interleave."""
    rng = np.random.default_rng(seed)
    pats = []
    for p in range(n_patterns):
        L = 1 if p % 7 == 3 else int(rng.integers(rows[0], rows[1] + 1))
        root, first = 0, int(rng.integers(1, n_ms))
        seq = [(root, first, int(rng.integers(0, n_if)))]
        called = [first]
        for _ in range(L - 1):
            um = called[int(rng.integers(0, len(called)))]
            dm = um if rng.random() < 0.08 else int(rng.integers(1, n_ms))            # self loops
            seq.append((um, dm, int(rng.integers(0, n_if))))
            called.append(dm)
        pats.append(np.array(seq, dtype=np.int64))
    entry_ids = np.sort(rng.choice(np.arange(2, 40), size=n_entries, replace=False)) * 3     # ids with gaps
    ent_pats = [list(rng.choice(n_patterns, size=int(rng.integers(2, 6)), replace=False)) for _ in range(n_entries)]
    ent_pats[1].append(int(ent_pats[0][0]))                                         # one pattern under two entries
    traceids = rng.choice(np.arange(10, 50 * n_traces), size=n_traces, replace=False).astype(np.int64) + traceid_base
    cols = {k: [] for k in ("traceid", "timestamp", "rpcid", "um", "dm", "interface", "rpctype", "rt", "entryid")}
    for i, tid in enumerate(traceids):
        e = int(rng.integers(0, n_entries))
        seq = pats[int(ent_pats[e][int(rng.integers(0, len(ent_pats[e])))])]
        n = len(seq)
        bucket = 30000 * int(rng.integers(1, 6))
        t0 = bucket + int(rng.choice([-2, -1, 0, 1, 5000, 20000])) if i % 5 == 0 else bucket + int(rng.integers(0, 29000))
        ts = t0 + np.concatenate([[0], np.sort(rng.integers(0, 900, size=n - 1))]).astype(np.int64)
        rt = rng.integers(1, 400, size=n) * np.where(rng.random(n) < 0.5, -1, 1)
        rt[0] = 1000 + int(rng.integers(0, 500))                                    # root: the largest |rt|
        rpcid = rng.permutation(n).astype(np.int64) + int(rng.integers(0, 1000))
        if n > 3 and rng.random() < 0.5:
            rpcid[int(rng.integers(2, n))] = rpcid[1]                                # repeated rpcid
        cols["traceid"].append(np.full(n, tid))
        cols["timestamp"].append(ts)
        cols["rpcid"].append(rpcid)
        cols["um"].append(seq[:, 0])
        cols["dm"].append(seq[:, 1])
        cols["interface"].append(seq[:, 2])
        cols["rpctype"].append(rng.integers(0, n_rpc, size=n))
        cols["rt"].append(rt)
        cols["entryid"].append(np.full(n, entry_ids[e]))
    table = {k: np.concatenate(v).astype(np.int64) for k, v in cols.items()}
    order = np.argsort(table["timestamp"], kind="stable")                           # get_df sorts by timestamp
    table = {k: v[order] for k, v in table.items()}
    buckets = np.unique(table["timestamp"] // 30000 * 30000)
    res_ts, res_ms = np.repeat(buckets, n_ms), np.tile(np.arange(n_ms, dtype=np.int64), len(buckets))
    resource = {"timestamp": res_ts, "msname": res_ms}
    vals = rng.random((len(res_ts), len(RESOURCE_COLUMNS)))
    for j, c in enumerate(RESOURCE_COLUMNS):
        resource[c] = vals[:, j]
    return table, resource
