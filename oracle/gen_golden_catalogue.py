"""Generates tests/golden/ref_catalogue.npz by RUNNING THE REFERENCE's preprocess.py main() (build container only:
needs /root/reference and pandas).

It writes synthetic.make_processed_tables(SEED) as processed/processed_df.csv + processed_resource_df.csv into a
temporary directory and runs main() there (loaded by path, as gen_golden_pert.py loads misc.py; nothing is copied).
Two settings make main() run under pandas 3: the legacy object dtype for strings (the string dtype breaks
map_consecutive_ids' ``df[:] = codes`` at preprocess.py:95), and ``interface`` before ``rpctype`` in the table (the
negative-stride view of misc.py:178, see gen_golden_pert.py).
Stored: the input table (``in_*``), tr2data (``tr_*``, dict order), entry2runtimes as a CSR (``ent_*``), and both
runtime2*graph maps in insertion order (``span_*`` / ``pert_*``: keys, occurrences, num_nodes and the concatenated
tensors with node / edge offsets), plus the Python type names of the tr2data values.
Usage:  python oracle/gen_golden_catalogue.py
"""
import contextlib
import importlib.util
import io
import os
import sys
import tempfile
import warnings

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from pert_gnn_kdd23_b200.synthetic import make_processed_tables  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden", "ref_catalogue.npz")
REF = "/root/reference"
SEED, N_TRACES = 5, 300
COLS = ("traceid", "timestamp", "rpcid", "um", "interface", "dm", "rpctype", "rt", "entryid")


def run_reference_main(table, resource):
    import pandas as pd
    import torch
    from joblib import load

    pd.set_option("future.infer_string", False)
    warnings.simplefilter("ignore")
    cwd = os.getcwd()
    sys.path.insert(0, REF)
    try:
        with tempfile.TemporaryDirectory() as d:
            os.makedirs(os.path.join(d, "processed"))
            pd.DataFrame({c: table[c] for c in COLS}).to_csv(os.path.join(d, "processed", "processed_df.csv"),
                                                           index=False)
            pd.DataFrame(resource).to_csv(os.path.join(d, "processed", "processed_resource_df.csv"), index=False)
            os.chdir(d)
            spec = importlib.util.spec_from_file_location("_ref_preprocess", os.path.join(REF, "preprocess.py"))
            mod = importlib.util.module_from_spec(spec)
            spec.loader.exec_module(mod)
            with contextlib.redirect_stdout(io.StringIO()), contextlib.redirect_stderr(io.StringIO()):
                mod.main()
            p = os.path.join(d, "processed")
            return (torch.load(os.path.join(p, "tr2data.pt"), weights_only=False),
                    load(os.path.join(p, "entry2runtimes.joblib")),
                    torch.load(os.path.join(p, "runtime2spangraph_map.pt"), weights_only=False),
                    torch.load(os.path.join(p, "runtime2pertgraph_map.pt"), weights_only=False))
    finally:
        os.chdir(cwd)
        sys.path.remove(REF)


def _graph_map(prefix, m):
    keys = list(m)
    out = {f"{prefix}_keys": np.array(keys, dtype=np.int64),
           f"{prefix}_occurences": np.array([m[k]["occurences"] for k in keys], dtype=np.int64),
           f"{prefix}_num_nodes": np.array([m[k]["num_nodes"] for k in keys], dtype=np.int64)}
    nptr, eptr = [0], [0]
    for k in keys:
        nptr.append(nptr[-1] + m[k]["ms_id"].shape[0])
        eptr.append(eptr[-1] + m[k]["edge_index"].shape[1])
    out[f"{prefix}_node_ptr"], out[f"{prefix}_edge_ptr"] = np.array(nptr), np.array(eptr)
    for f in ("ms_id", "node_depth"):
        out[f"{prefix}_{f}"] = np.concatenate([m[k][f].numpy().reshape(-1) for k in keys]).astype(np.int64)
    out[f"{prefix}_edge_index"] = np.concatenate([m[k]["edge_index"].numpy() for k in keys], axis=1).astype(np.int64)
    out[f"{prefix}_edge_attr"] = np.concatenate([m[k]["edge_attr"].numpy() for k in keys], axis=0).astype(np.int64)
    return out


def main():
    table, resource = make_processed_tables(SEED, N_TRACES)
    tr2data, e2r, span, pert = run_reference_main(table, resource)
    out = {f"in_{c}": table[c] for c in table}
    keys = list(tr2data)
    out["tr_keys"] = np.array(keys, dtype=np.int64)
    for f in ("entry_id", "runtime_id", "timestamp", "y"):
        out[f"tr_{f}"] = np.array([int(tr2data[k][f]) for k in keys], dtype=np.int64)
    v0 = tr2data[keys[0]]
    out["tr_types"] = np.array([type(keys[0]).__name__] + [type(v0[f]).__name__ for f in
                                                           ("entry_id", "runtime_id", "timestamp", "y")])
    out["tr_y_dtype"] = np.array(str(v0["y"].dtype))
    ents = list(e2r)
    out["ent_keys"] = np.array(ents, dtype=np.int64)
    out["ent_ptr"] = np.concatenate([[0], np.cumsum([len(e2r[e]) for e in ents])]).astype(np.int64)
    out["ent_runtime_id"] = np.array([r for e in ents for r in e2r[e]], dtype=np.int64)
    out["ent_prob"] = np.array([p for e in ents for p in e2r[e].values()], dtype=np.float64)
    out.update(_graph_map("span", span))
    out.update(_graph_map("pert", pert))
    np.savez_compressed(OUT, **out)
    print("wrote", OUT, os.path.getsize(OUT), "bytes;", len(keys), "traces,", len(span), "patterns")


if __name__ == "__main__":
    main()
