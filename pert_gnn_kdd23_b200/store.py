"""Device-resident pattern store + on-device batch assembly (SURVEY.md section 8f rows N1 and N4).

The reference assembles every sample on the host (``get_entry_data``, pert_gnn.py:134-173: pandas feature join
``get_x`` :40-67, cached per-pattern tensor builders :77-131), caches the resulting 100k-element ``data_list``
("10+hrs", README.md:12), collates batches with PyG's DataLoader (:201-209) and rebuilds the per-node pattern
probability on the host every step with B tiny H2D copies (:220-230).

``PatternStore`` keeps the reference's artefacts (``runtime2graph``, ``entry2runtimes``, ``resource_df``, ``tr2data`` --
what pert_gnn.py:297-305 loads) resident in HBM in concatenated int32/int64/float32 arrays; ``assemble(trace_ids)``
turns a list of trace ids (8 bytes per graph of H2D traffic instead of ~33 KB) into the collated device ``Batch`` with
4 kernel launches (csrc/store.cu) -- the tensors are bit-identical to ``Batch.from_data_list([get_entry_data(...)])`` +
``transform_pattern_probs`` (tests/test_store.py checks them against the reference's own outputs,
tests/golden/ref_loop.npz).  No CPU fallback: the store lives on a CUDA device.
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import _lib
from .data import Batch

I32, I64, P = C.c_int32, C.c_longlong, C.c_void_p


class _PertStore(C.Structure):
    _fields_ = [("n_pat", I32), ("n_ent", I32), ("n_res", I32), ("n_ms", I32), ("attr_cols", I32),
                ("n_traces", I64),
                ("pat_nptr", P), ("pat_eptr", P), ("pat_ms", P), ("pat_depth", P), ("pat_last", P), ("pat_src", P),
                ("pat_dst", P), ("pat_attr", P), ("ent_ptr", P), ("ent_pat", P), ("ent_prob", P), ("ent_nodes", P),
                ("ent_edges", P), ("res_keys", P), ("res_vals", P), ("ms_has_res", P), ("trace_entry", P),
                ("trace_ts", P), ("trace_y", P)]


class _PertBatchOut(C.Structure):
    _fields_ = [(k, P) for k in ("x", "cat_X", "node_depth", "pattern_num_nodes", "rt_probs", "batch", "edge_index",
                                 "edge_attr", "entry_id", "y", "ptr", "pattern_probs")]


def _last_occurrence_flags(all_ms, nptr):
    """flags[i] = 1 iff node i is the LAST node of its microservice inside its pattern (patterns = nptr slices)."""
    n_all = int(all_ms.shape[0])
    flags = np.zeros(n_all, dtype=np.uint8)
    if n_all:
        pid = np.repeat(np.arange(len(nptr) - 1, dtype=np.int64), np.diff(nptr))
        lo = int(all_ms.min())
        key = pid * (int(all_ms.max()) - lo + 1) + (all_ms - lo)
        _, first_rev = np.unique(key[::-1], return_index=True)
        flags[n_all - 1 - first_rev] = 1
    return flags


class _BulkPatterns:
    """Concatenated host arrays of many patterns (PatternStore.from_graphs)."""

    def __init__(self, rt_ids, node_ptr, edge_ptr, ms_id, node_depth, edge_index, edge_attr):
        self.rt_ids, self.node_ptr, self.edge_ptr = rt_ids, node_ptr, edge_ptr
        self.ms_id, self.node_depth, self.edge_index, self.edge_attr = ms_id, node_depth, edge_index, edge_attr


class _EntryCSR:
    """entry2runtimes as arrays over entry ids 0..n_ent-1 (PatternStore.from_catalogue): ent_ptr [n_ent+1], ent_pat
    (pattern index), ent_prob (float64)."""

    def __init__(self, ent_ptr, ent_pat, ent_prob):
        self.ent_ptr, self.ent_pat, self.ent_prob = ent_ptr, ent_pat, ent_prob


class _TraceArrays:
    """tr2data as arrays in its dict order (PatternStore.from_catalogue): keys, entry, ts, y."""

    def __init__(self, keys, entry, ts, y):
        self.keys, self.entry, self.ts, self.y = keys, entry, ts, y


class PatternStore:
    """Patterns, entries, resource table and traces on one CUDA device."""

    def __init__(self, runtime2graph, entry2runtimes, resource_index, resource_values, tr2data, device, n_ms=None):
        dev = torch.device(device)
        if dev.type != "cuda":
            raise _lib.PertGnnError("PatternStore lives on a CUDA device (no CPU fallback for the hot path)")
        self.device = dev
        # ---- patterns, in the dict order of runtime2graph (or the bulk arrays of pertgraph.PertGraphs, see from_graphs)
        if isinstance(runtime2graph, _BulkPatterns):
            bp = runtime2graph
            self.rt_ids = list(bp.rt_ids)
            nptr, eptr = bp.node_ptr.astype(np.int64), bp.edge_ptr.astype(np.int64)
            ms = [bp.ms_id.astype(np.int64)]
            depth = [bp.node_depth.astype(np.int64)]
            src, dst = [bp.edge_index[0].astype(np.int32)], [bp.edge_index[1].astype(np.int32)]
            attr = [bp.edge_attr.astype(np.int64)]
            cols = bp.edge_attr.shape[1]
        else:
            self.rt_ids = list(runtime2graph.keys())
            nptr, eptr = [0], [0]
            ms, depth, src, dst, attr = [], [], [], [], []
            cols = None
            for rt in self.rt_ids:
                g = runtime2graph[rt]
                n = int(g["num_nodes"])
                # patterns may be CUDA tensors (pertgraph.PertGraphs.pattern): the host copy sizes batches and finds the
                # last occurrence of every microservice; for many patterns use PatternStore.from_graphs (one bulk copy)
                m = g["ms_id"].reshape(-1).to(torch.int64).cpu().numpy()
                assert m.shape[0] == n
                ei = g["edge_index"].cpu().numpy()
                ea = g["edge_attr"].cpu().numpy()
                cols = ea.shape[1] if cols is None else cols
                assert ea.shape[1] == cols
                nptr.append(nptr[-1] + n)
                eptr.append(eptr[-1] + ei.shape[1])
                ms.append(m)
                depth.append(g["node_depth"].reshape(-1).to(torch.int64).cpu().numpy())
                src.append(ei[0].astype(np.int32))
                dst.append(ei[1].astype(np.int32))
                attr.append(ea.astype(np.int64))
        rt_index = {rt: i for i, rt in enumerate(self.rt_ids)}
        nptr, eptr = np.asarray(nptr, dtype=np.int64), np.asarray(eptr, dtype=np.int64)
        # get_x's dict ms2nid keeps the LAST node of every microservice of a pattern (pert_gnn.py:54-65): vectorised as
        # the first occurrence of (pattern, ms) in the reversed node list
        all_ms = np.concatenate(ms) if ms else np.zeros(0, dtype=np.int64)
        last_flags = _last_occurrence_flags(all_ms, nptr)
        last = [last_flags]
        self.attr_cols = int(cols)
        pat_nodes = np.diff(nptr)
        pat_edges = np.diff(eptr)
        # ---- entries, in the dict order of entry2runtimes[entry] (get_all_runtimes_id_probs, pert_gnn.py:70-74)
        if isinstance(entry2runtimes, _EntryCSR):
            ec = entry2runtimes
            n_ent = len(ec.ent_ptr) - 1
            ent_ptr, ent_pat, ent_prob = ec.ent_ptr, ec.ent_pat, ec.ent_prob
            pe = np.repeat(np.arange(n_ent), np.diff(ent_ptr))
            ent_nodes = np.bincount(pe, weights=pat_nodes[ent_pat], minlength=n_ent).astype(np.int32)
            ent_edges = np.bincount(pe, weights=pat_edges[ent_pat], minlength=n_ent).astype(np.int32)
        else:
            n_ent = max(entry2runtimes.keys()) + 1
            ent_ptr, ent_pat, ent_prob = [0], [], []
            ent_nodes, ent_edges = np.zeros(n_ent, dtype=np.int32), np.zeros(n_ent, dtype=np.int32)
            for e in range(n_ent):
                for rt, pr in entry2runtimes.get(e, {}).items():
                    k = rt_index[rt]
                    ent_pat.append(k)
                    ent_prob.append(pr)
                    ent_nodes[e] += pat_nodes[k]
                    ent_edges[e] += pat_edges[k]
                ent_ptr.append(len(ent_pat))
        res_ms = np.array([m for _, m in resource_index], dtype=np.int64)
        res_ts = np.array([t for t, _ in resource_index], dtype=np.int64)
        self.n_ms = int(n_ms if n_ms is not None else max(int(all_ms.max(initial=0)), int(res_ms.max(initial=0))) + 1)
        keys = res_ts * self.n_ms + res_ms
        order = np.argsort(keys, kind="stable")
        has = np.zeros(self.n_ms, dtype=np.uint8)
        has[res_ms] = 1                                          # ms_with_resources (pert_gnn.py:138)
        # ---- traces, in the dict order of tr2data (get_data_list, pert_gnn.py:176-188)
        if isinstance(tr2data, _TraceArrays):
            self.trace_keys = tr2data.keys
            t_ent, t_ts, t_y = tr2data.entry.astype(np.int32), tr2data.ts, tr2data.y
        else:
            self.trace_keys = list(tr2data.keys())
            t_ent = np.array([int(tr2data[k]["entry_id"]) for k in self.trace_keys], dtype=np.int32)
            t_ts = np.array([int(tr2data[k]["timestamp"]) for k in self.trace_keys], dtype=np.int64)
            t_y = np.array([int(tr2data[k]["y"]) for k in self.trace_keys], dtype=np.int64)
        # host copies used to size the outputs without a device sync
        self._h_ent_nodes, self._h_ent_edges = ent_nodes.astype(np.int64), ent_edges.astype(np.int64)
        self._h_ent_pats = np.diff(np.array(ent_ptr)).astype(np.int64)
        self._h_trace_entry = t_ent.astype(np.int64)

        def up(a, dtype):
            return torch.from_numpy(np.ascontiguousarray(a, dtype=dtype)).to(dev)

        cat = lambda xs, dt: np.concatenate(xs).astype(dt) if xs else np.zeros(0, dtype=dt)   # noqa: E731
        self.t = {
            "pat_nptr": up(nptr, np.int32), "pat_eptr": up(eptr, np.int32), "pat_ms": up(cat(ms, np.int64), np.int64),
            "pat_depth": up(cat(depth, np.int64), np.int64), "pat_last": up(cat(last, np.uint8), np.uint8),
            "pat_src": up(cat(src, np.int32), np.int32), "pat_dst": up(cat(dst, np.int32), np.int32),
            "pat_attr": up(np.concatenate(attr, axis=0) if attr else np.zeros((0, 2)), np.int64),
            "ent_ptr": up(ent_ptr, np.int32), "ent_pat": up(ent_pat, np.int32),
            # torch.tensor(python floats, dtype=torch.float) of the reference == float64 -> float32 rounding
            "ent_prob": up(np.array(ent_prob, dtype=np.float64).astype(np.float32), np.float32),
            "ent_nodes": up(ent_nodes, np.int32), "ent_edges": up(ent_edges, np.int32),
            "res_keys": up(keys[order], np.int64),
            "res_vals": up(np.asarray(resource_values, dtype=np.float64)[order].astype(np.float32), np.float32),
            "ms_has_res": up(has, np.uint8), "trace_entry": up(t_ent, np.int32), "trace_ts": up(t_ts, np.int64),
            "trace_y": up(t_y, np.int64),
        }
        d = _PertStore()
        d.n_pat, d.n_ent, d.n_res, d.n_ms, d.attr_cols = len(self.rt_ids), n_ent, int(keys.shape[0]), self.n_ms, \
            self.attr_cols
        d.n_traces = len(self.trace_keys)
        for k, v in self.t.items():
            setattr(d, k, v.data_ptr())
        self.desc = d
        self.status = torch.zeros(1, dtype=torch.int32, device=dev)

    @classmethod
    def from_graphs(cls, graphs, runtime_ids, entry2runtimes, resource_index, resource_values, tr2data, device=None,
                    n_ms=None):
        """Patterns straight from ``pertgraph.build_pert_graphs`` / ``build_span_graphs`` (``graphs``: PertGraphs;
        ``runtime_ids[i]`` names pattern i): ONE device->host copy of the concatenated tensors instead of one per
        pattern, no per-pattern Python work."""
        dev = torch.device(device) if device is not None else graphs.ms_id.device
        bp = _BulkPatterns(list(runtime_ids), np.asarray(graphs.node_ptr), np.asarray(graphs.edge_ptr),
                           graphs.ms_id.cpu().numpy().reshape(-1), graphs.node_depth.cpu().numpy().reshape(-1),
                           graphs.edge_index.cpu().numpy(), graphs.edge_attr.cpu().numpy())
        assert len(bp.rt_ids) == len(bp.node_ptr) - 1
        return cls(bp, entry2runtimes, resource_index, resource_values, tr2data, dev, n_ms=n_ms)

    @classmethod
    def from_catalogue(cls, cat, graphs, resource_index, resource_values, device=None, n_ms=None):
        """Store of a ``catalogue.Catalogue`` (``graphs``: ``cat.graphs(kind)``) without per-trace or per-entry Python
        dicts: the same device arrays as ``PatternStore(*cat.to_reference(kind), resource_index, resource_values,
        ...)`` (traces in tr2data order, patterns in runtime2graph order, entries by id)."""
        h = {k: getattr(cat, k).cpu().numpy() for k in ("traceid", "entry", "timestamp", "y", "pat_runtime_id",
                                                         "entries", "ent_ptr", "ent_runtime_id", "ent_prob")}
        pos = np.empty(len(h["pat_runtime_id"]), dtype=np.int64)
        pos[h["pat_runtime_id"]] = np.arange(len(pos))                 # runtime id -> pattern index
        n_ent = int(h["entries"].max()) + 1
        counts = np.zeros(n_ent, dtype=np.int64)
        counts[h["entries"]] = np.diff(h["ent_ptr"])
        ent_ptr = np.concatenate([[0], np.cumsum(counts)]).astype(np.int64)
        entries = _EntryCSR(ent_ptr, pos[h["ent_runtime_id"]], h["ent_prob"])
        traces = _TraceArrays(h["traceid"].tolist(), h["entry"], h["timestamp"], h["y"])
        dev = torch.device(device) if device is not None else cat.device
        bp = _BulkPatterns(h["pat_runtime_id"].tolist(), np.asarray(graphs.node_ptr), np.asarray(graphs.edge_ptr),
                           graphs.ms_id.cpu().numpy().reshape(-1), graphs.node_depth.cpu().numpy().reshape(-1),
                           graphs.edge_index.cpu().numpy(), graphs.edge_attr.cpu().numpy())
        assert len(bp.rt_ids) == len(bp.node_ptr) - 1
        return cls(bp, entries, resource_index, resource_values, traces, dev, n_ms=n_ms)

    @classmethod
    def from_artifacts(cls, art, device):
        """``art``: dict with the reference's artefacts (synthetic.make_trace_artifacts schema; with ``graphs`` +
        ``runtime_ids`` -- synthetic.make_pert_artifacts -- the patterns are taken from the device-resident PertGraphs)."""
        if art.get("graphs") is not None:
            return cls.from_graphs(art["graphs"], art["runtime_ids"], art["entry2runtimes"], art["resource_index"],
                                   art["resource_values"], art["tr2data"], device, n_ms=art.get("n_ms"))
        return cls(art["runtime2graph"], art["entry2runtimes"], art["resource_index"], art["resource_values"],
                   art["tr2data"], device, n_ms=art.get("n_ms"))

    def __len__(self):
        return len(self.trace_keys)

    @property
    def resident_bytes(self):
        return sum(v.numel() * v.element_size() for v in self.t.values())

    def sizes(self, trace_ids):
        """(N, E, P) of a batch from the host copies -- no device sync."""
        ent = self._h_trace_entry[np.asarray(trace_ids, dtype=np.int64)]
        return int(self._h_ent_nodes[ent].sum()), int(self._h_ent_edges[ent].sum()), int(self._h_ent_pats[ent].sum())

    @_lib.on_device_of
    def assemble(self, trace_ids, ids_device=None):
        """-> device ``Batch`` of the traces ``trace_ids`` (sequence of ints into the store's trace table).
        ``ids_device``: the same ids already on the device (int64) -- e.g. a slice of a resident epoch permutation --
        to skip even the 8-byte-per-graph H2D copy."""
        ids = np.asarray(trace_ids, dtype=np.int64)
        B = int(ids.shape[0])
        N, E, Pn = self.sizes(ids)
        dev = self.device
        if ids_device is None:
            ids_device = torch.from_numpy(ids).to(dev, non_blocking=True)
        f32, i64 = torch.float32, torch.int64
        out = {
            "x": torch.empty(N, 9, dtype=f32, device=dev), "edge_index": torch.empty(2, E, dtype=i64, device=dev),
            "edge_attr": torch.empty(E, self.attr_cols, dtype=i64, device=dev),
            "cat_X": torch.empty(N, 1, dtype=i64, device=dev), "node_depth": torch.empty(N, 1, dtype=i64, device=dev),
            "pattern_num_nodes": torch.empty(N, 1, dtype=f32, device=dev),
            "pattern_probs": torch.empty(Pn, 1, dtype=f32, device=dev),
            "entry_id": torch.empty(B, dtype=i64, device=dev), "y": torch.empty(B, dtype=i64, device=dev),
            "rt_probs": torch.empty(N, 1, dtype=f32, device=dev), "batch": torch.empty(N, dtype=i64, device=dev),
            "ptr": torch.empty(B + 1, dtype=i64, device=dev),
        }
        offsets = torch.empty(3 * (B + 1), dtype=torch.int32, device=dev)
        o = _PertBatchOut()
        for k in ("x", "cat_X", "node_depth", "pattern_num_nodes", "rt_probs", "batch", "edge_index", "edge_attr",
                  "entry_id", "y", "ptr", "pattern_probs"):
            setattr(o, k, out[k].data_ptr())
        rc = _lib.lib().pert_store_assemble(C.byref(self.desc), ids_device.data_ptr(), B, N, E, offsets.data_ptr(),
                                            C.byref(o), self.status.data_ptr(), _lib.stream())
        _lib.check(rc, "pert_store_assemble")
        from . import ops

        ops.LAUNCHES["n"] += 4
        b = Batch()
        b._store.update(out)
        object.__setattr__(b, "_num_graphs", B)
        object.__setattr__(b, "_keepalive", (ids_device, offsets))
        return b

    def check(self):
        """Synchronising check of the status word (trace id out of range / missing (timestamp, ms) row)."""
        code = int(self.status.item())
        if code != 0:
            _lib.check(code, "pert_store_assemble")


class StoreLoader:
    """DataLoader-shaped iterator over a PatternStore: yields device batches assembled on the GPU.
    ``torch_geometric.loader.DataLoader(data_list, batch_size, shuffle)`` look-alike (``len(loader.dataset)``, iteration)
    for the part of the reference loop that consumes batches (pert_gnn.py:219, :260)."""

    def __init__(self, store: PatternStore, trace_ids, batch_size, shuffle=False, generator=None):
        self.store, self.batch_size, self.shuffle, self.generator = store, int(batch_size), shuffle, generator
        self.dataset = list(trace_ids)

    def __len__(self):
        return -(-len(self.dataset) // self.batch_size)

    def __iter__(self):
        ids = np.asarray(self.dataset, dtype=np.int64)
        if self.shuffle:
            perm = torch.randperm(len(ids), generator=self.generator).numpy()
            ids = ids[perm]
        for i in range(0, len(ids), self.batch_size):
            yield self.store.assemble(ids[i:i + self.batch_size])
