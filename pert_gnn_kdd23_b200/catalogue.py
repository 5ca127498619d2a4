"""Trace catalogue on the GPU: what preprocess.py:main() (:269-375) derives from the integer-coded span table.

Input: the ``processed_df`` table (int64 columns ``traceid, timestamp, rpcid, um, dm, interface, rpctype, rt,
entryid``) in file order.  Output (``Catalogue``, arrays on the device):
  * per trace, in the reference's ``tr2data`` order (entry ascending, then traceid ascending; :295-309):
    ``traceid``, ``entry``, ``runtime_id``, ``timestamp`` (floor(min timestamp / 30000) * 30000, :39) and ``y``
    (max |rt|, :290-292).  Two traces share a runtime id iff their raw rows give the same (um, dm, interface) sequence
    in file order; ids are numbered by first appearance in traceid order (factorize over groupby, :280-293);
  * per pattern, in ``runtime2graph`` insertion order (the order the representatives are met, :317-367):
    ``pat_runtime_id``, ``pat_trace`` (representative: first trace showing it in tr2data order, as a position into the
    traceid-sorted traces), ``pat_traceid``, ``pat_occurrences``;
  * entry CSR (``entry2runtimes``, :310-316 + :371-375): ``entries[E]`` ascending, ``ent_ptr[E+1]`` into
    ``ent_runtime_id`` (patterns in order of first appearance inside the entry) and ``ent_prob`` (float64,
    count / total, bit-identical to Python's int / int).
The hot path is csrc/catalogue.cu (one warp per trace over the grouped rows, exact dedup, ids / counts kernels);
torch's stable sorts, scans and ``nonzero`` are the plumbing between them.  The host syncs are those that size
outputs (trace, pattern, entry and pair counts) and one per dedup round (whether a member differs from its head).

Not reproduced: the reference raises ``KeyError`` when a representative's timestamp bucket lacks resource rows
(find_most_recent_fts / get_node_features); the graphs it stores do not depend on those rows.  A trace whose rows
carry different ``entryid`` values is rejected (the reference's get_df makes entryid a function of traceid).
"""
from __future__ import annotations

import numpy as np
import torch

from . import _lib
from . import pertgraph

COLUMNS = ("traceid", "timestamp", "rpcid", "um", "dm", "interface", "rpctype", "rt", "entryid")
MAX_REKEY_ROUNDS = 64

# Test hook (like SAGEDeterministic._capture): set to a dict before build_catalogue; ``hash_mask`` in it masks every
# sequence hash (forcing collisions), and the build writes ``rekey_rounds`` / ``mismatches`` back into it.
_hook = None


def _check_table(table):
    """Host-side argument checks, before any CUDA call."""
    missing = [c for c in COLUMNS if c not in table]
    if missing:
        raise KeyError(f"span table lacks column(s) {missing}; needs {list(COLUMNS)}")
    n = None
    for c in COLUMNS:
        v = table[c]
        dt = v.dtype if torch.is_tensor(v) else np.asarray(v).dtype
        if dt not in (torch.int64, np.dtype(np.int64)):
            raise TypeError(f"column {c!r} has dtype {dt}; the span table is int64")
        shape = tuple(v.shape) if torch.is_tensor(v) else np.asarray(v).shape
        if len(shape) != 1:
            raise ValueError(f"column {c!r} must be 1-D, got shape {shape}")
        if n is None:
            n = shape[0]
        elif shape[0] != n:
            raise ValueError(f"column {c!r} has {shape[0]} rows, {COLUMNS[0]!r} has {n}")
    if not n:
        raise ValueError("empty span table")


def _as_device_columns(table, dev):
    out = {}
    for c in COLUMNS:
        v = table[c]
        t = v if torch.is_tensor(v) else torch.from_numpy(np.ascontiguousarray(v))
        out[c] = t.to(dev, non_blocking=True).contiguous()
    return out


def _head_positions(sorted_key):
    """Sorted position of the first element of every run of equal keys."""
    n = sorted_key.shape[0]
    flag = torch.empty(n, dtype=torch.int64, device=sorted_key.device)
    mark = torch.empty_like(flag)
    _lib.call("pert_catalogue_run_flags", _lib.ptr(sorted_key), n, _lib.ptr(flag), _lib.ptr(mark), _lib.stream())
    return torch.cummax(mark, 0).values


def _run_starts(sorted_key):
    n = sorted_key.shape[0]
    flag = torch.empty(n, dtype=torch.int64, device=sorted_key.device)
    _lib.call("pert_catalogue_run_flags", _lib.ptr(sorted_key), n, _lib.ptr(flag), None, _lib.stream())
    return flag, torch.nonzero(flag).reshape(-1)                 # nonzero: a sizing sync


def build_catalogue(table, device="cuda"):
    """``table``: dict of int64 numpy arrays or CUDA tensors (``COLUMNS``), rows in file order.  -> ``Catalogue``."""
    _check_table(table)
    dev = torch.device(device)
    if dev.type != "cuda":
        raise _lib.PertGnnError("build_catalogue needs a CUDA device (no CPU fallback)")
    hook = _hook
    mask = int(hook.get("hash_mask", (1 << 64) - 1)) if isinstance(hook, dict) else (1 << 64) - 1
    with torch.cuda.device(dev):
        cols = _as_device_columns(table, dev)
        R = int(cols["traceid"].shape[0])
        st = _lib.stream()
        i64 = dict(dtype=torch.int64, device=dev)
        # ---- group rows by traceid (stable: file order inside a trace), trace positions = ascending traceid
        tid_sorted, perm = torch.sort(cols["traceid"], stable=True)
        _, starts = _run_starts(tid_sorted)
        T = int(starts.shape[0])
        row_ptr = torch.empty(T + 1, **i64)
        row_ptr[:T] = starts
        row_ptr[T] = R
        traceid = tid_sorted[starts]
        um, dm, itf = cols["um"], cols["dm"], cols["interface"]
        nrows, key, y, ts_bucket, entry = (torch.empty(T, **i64) for _ in range(5))
        status = torch.zeros(1, dtype=torch.int32, device=dev)
        _lib.call("pert_catalogue_summary", _lib.ptr(perm), _lib.ptr(row_ptr), T, _lib.ptr(um), _lib.ptr(dm),
                  _lib.ptr(itf), _lib.ptr(cols["rt"]), _lib.ptr(cols["timestamp"]), _lib.ptr(cols["entryid"]), 0, mask,
                  _lib.ptr(nrows), _lib.ptr(key), _lib.ptr(y), _lib.ptr(ts_bucket), _lib.ptr(entry), _lib.ptr(status),
                  st)
        # ---- exact dedup: sort by (key, position), compare every run member with its head, re-key the ones that differ
        mismatch = torch.empty(T, dtype=torch.int32, device=dev)
        n_mis = torch.empty(1, **i64)
        rounds, mismatches = 0, 0
        while True:
            skey, order = torch.sort(key, stable=True)
            head = _head_positions(skey)
            _lib.call("pert_catalogue_verify", _lib.ptr(order), _lib.ptr(head), T, _lib.ptr(perm), _lib.ptr(row_ptr),
                      _lib.ptr(um), _lib.ptr(dm), _lib.ptr(itf), _lib.ptr(mismatch), _lib.ptr(n_mis), st)
            flags = torch.cat([n_mis, status.to(torch.int64)]).cpu()
            if rounds == 0 and int(flags[1]) != 0:
                raise _lib.PertGnnError("build_catalogue: a trace's rows carry different entryid values")
            if int(flags[0]) == 0:
                break
            mismatches += int(flags[0])
            rounds += 1
            if rounds > MAX_REKEY_ROUNDS:
                raise _lib.PertGnnError("build_catalogue: sequence hashes did not separate the patterns")
            _lib.call("pert_catalogue_rekey", _lib.ptr(perm), _lib.ptr(row_ptr), T, _lib.ptr(um), _lib.ptr(dm),
                      _lib.ptr(itf), _lib.ptr(mismatch), rounds, mask, _lib.ptr(key), st)
        if isinstance(hook, dict):
            hook["rekey_rounds"], hook["mismatches"] = rounds, mismatches
        # ---- runtime ids in factorize order (first trace of each pattern in traceid order, scanned)
        canon, first = torch.empty(T, **i64), torch.empty(T, **i64)
        _lib.call("pert_catalogue_canon", _lib.ptr(order), _lib.ptr(head), T, _lib.ptr(canon), _lib.ptr(first), st)
        first_incl = torch.cumsum(first, 0)
        rid = torch.empty(T, **i64)
        _lib.call("pert_catalogue_runtime_ids", _lib.ptr(canon), _lib.ptr(first_incl), T, _lib.ptr(rid), st)
        P = int(first_incl[-1])                                   # sizing sync
        # ---- (entry, traceid) order, representatives, occurrences, (entry, pattern) pairs
        ent_sorted, eorder = torch.sort(entry, stable=True)
        eflag, ent_start = _run_starts(ent_sorted)
        E = int(ent_start.shape[0])
        eidx = torch.cumsum(eflag, 0) - 1
        rep_epos, occ, pair_key = torch.empty(P, **i64), torch.empty(P, **i64), torch.empty(T, **i64)
        _lib.call("pert_catalogue_patterns", _lib.ptr(eorder), _lib.ptr(eidx), T, _lib.ptr(rid), P, _lib.ptr(rep_epos),
                  _lib.ptr(occ), _lib.ptr(pair_key), st)
        pk_sorted, pidx = torch.sort(pair_key, stable=True)
        _, pstart = _run_starts(pk_sorted)
        NP = int(pstart.shape[0])
        count, pfirst, pent, prid = (torch.empty(NP, **i64) for _ in range(4))
        _lib.call("pert_catalogue_pairs", _lib.ptr(pstart), NP, T, _lib.ptr(pidx), _lib.ptr(eorder), _lib.ptr(rid),
                  _lib.ptr(eidx), _lib.ptr(count), _lib.ptr(pfirst), _lib.ptr(pent), _lib.ptr(prid), st)
        q = torch.sort(pfirst).indices                            # distinct keys: entry-major, first appearance
        pent, count, prid = pent[q].contiguous(), count[q].contiguous(), prid[q].contiguous()
        prob = torch.empty(NP, dtype=torch.float64, device=dev)
        ent_ptr = torch.empty(E + 1, **i64)
        _lib.call("pert_catalogue_probs", _lib.ptr(pent), _lib.ptr(count), NP, _lib.ptr(ent_start), E, T,
                  _lib.ptr(prob), _lib.ptr(ent_ptr), st)
        po = torch.sort(rep_epos).indices                         # insertion order of runtime2graph
        pat_trace = eorder[rep_epos[po]]
        return Catalogue(
            traceid=traceid[eorder], entry=entry[eorder], runtime_id=rid[eorder], timestamp=ts_bucket[eorder],
            y=y[eorder], pat_runtime_id=po, pat_trace=pat_trace, pat_traceid=traceid[pat_trace],
            pat_occurrences=occ[po], entries=ent_sorted[ent_start], ent_ptr=ent_ptr, ent_runtime_id=prid,
            ent_prob=prob, columns=cols, perm=perm, row_ptr=row_ptr, rekey_rounds=rounds)


class Catalogue:
    """Device arrays of one span table's catalogue (see the module docstring for their order)."""

    def __init__(self, **arrays):
        rounds = arrays.pop("rekey_rounds")
        self._columns, self._perm, self._row_ptr = arrays.pop("columns"), arrays.pop("perm"), arrays.pop("row_ptr")
        for k, v in arrays.items():
            setattr(self, k, v)
        self.rekey_rounds = rounds
        self.device = self.traceid.device

    def __len__(self):
        return int(self.traceid.shape[0])

    @property
    def num_patterns(self):
        return int(self.pat_runtime_id.shape[0])

    @_lib.on_device_of
    def graphs(self, kind="span"):
        """``PertGraphs`` of the patterns (pattern order), built from the representatives' raw rows through
        ``pertgraph.clean_span_tables_flat`` (misc.py:87-105, :138-142) and ``build_pert_graphs_flat``."""
        lens = (self._row_ptr[1:] - self._row_ptr[:-1])[self.pat_trace]
        rp = torch.zeros(lens.shape[0] + 1, dtype=torch.int64, device=self.device)
        torch.cumsum(lens, 0, out=rp[1:])
        rp_h = rp.cpu().numpy()                                   # sizing sync
        n = int(rp_h[-1])
        within = torch.arange(n, device=self.device) - torch.repeat_interleave(rp[:-1], lens, output_size=n)
        rows = self._perm[torch.repeat_interleave(self._row_ptr[self.pat_trace], lens, output_size=n) + within]
        names = ("um", "dm", "rpcid", "rt", "timestamp", "interface", "rpctype")
        host = torch.stack([self._columns[c][rows] for c in names]).cpu().numpy()
        c = dict(zip(names, host))
        keep, new_ptr, roots = pertgraph.clean_span_tables_flat(c, rp_h)
        c["endTimestamp"] = c["timestamp"] + np.abs(c["rt"])
        flat = np.stack([c[k][keep] for k in pertgraph.COLUMNS])
        return pertgraph.build_pert_graphs_flat(flat, new_ptr, roots, self.device, kind=kind).check()

    def to_reference(self, kind="span", graphs=None):
        """-> (tr2data, entry2runtimes, runtime2graph) with the keys, orders and value types preprocess.py:main() saves
        (runtime2graph = its ``runtime2spangraph_map`` for kind "span", ``runtime2pertgraph_map`` for "pert"; PERT node
        numbering is pertgraph's canonical one).  ``graphs``: the result of ``graphs(kind)`` if already built."""
        h = {k: getattr(self, k).cpu().numpy() for k in ("traceid", "entry", "runtime_id", "timestamp", "y",
                                                           "pat_runtime_id", "pat_occurrences", "entries", "ent_ptr",
                                                           "ent_runtime_id", "ent_prob")}
        tr2data = {}
        for tid, e, r, ts, y in zip(*(h[k].tolist() for k in ("traceid", "entry", "runtime_id", "timestamp", "y"))):
            tr2data[tid] = {"entry_id": e, "runtime_id": r, "timestamp": np.int64(ts), "y": torch.tensor(y)}
        entry2runtimes = {}
        rids, probs, ptr = h["ent_runtime_id"].tolist(), h["ent_prob"].tolist(), h["ent_ptr"].tolist()
        for i, e in enumerate(h["entries"].tolist()):
            entry2runtimes[e] = dict(zip(rids[ptr[i]:ptr[i + 1]], probs[ptr[i]:ptr[i + 1]]))
        g = graphs if graphs is not None else self.graphs(kind)
        runtime2graph = {}
        for k, (rt, oc) in enumerate(zip(h["pat_runtime_id"].tolist(), h["pat_occurrences"].tolist())):
            p = g.pattern(k)
            runtime2graph[rt] = {"edge_index": p["edge_index"].cpu(), "ms_id": p["ms_id"].cpu(), "occurences": oc,
                                 "num_nodes": p["num_nodes"], "node_depth": p["node_depth"].cpu(),
                                 "edge_attr": p["edge_attr"].cpu()}
        return tr2data, entry2runtimes, runtime2graph
