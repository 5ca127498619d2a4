"""Trace catalogue (pert_gnn_kdd23_b200/catalogue.py, csrc/catalogue.cu) against the reference's own preprocess.py
main() outputs (tests/golden/ref_catalogue.npz, oracle/gen_golden_catalogue.py) and the numpy oracle
(oracle/catalogue_oracle.py)."""
import os

import numpy as np
import pytest
import torch

from oracle import catalogue_oracle as CO
from oracle import pert_graph_oracle as O
from pert_gnn_kdd23_b200 import catalogue as C
from pert_gnn_kdd23_b200 import pertgraph
from pert_gnn_kdd23_b200.synthetic import make_processed_tables

GOLDEN = os.path.join(os.path.dirname(__file__), "golden", "ref_catalogue.npz")


def _golden():
    z = np.load(GOLDEN)
    return z, {k[3:]: z[k] for k in z.files if k.startswith("in_")}


def _fixture_graph(z, prefix, k):
    n0, n1 = z[f"{prefix}_node_ptr"][k:k + 2]
    e0, e1 = z[f"{prefix}_edge_ptr"][k:k + 2]
    return (z[f"{prefix}_ms_id"][n0:n1], z[f"{prefix}_edge_index"][:, e0:e1], z[f"{prefix}_edge_attr"][e0:e1],
            z[f"{prefix}_node_depth"][n0:n1].reshape(-1, 1))


def _fixture_dicts(z):
    """The reference's tr2data / entry2runtimes / runtime2spangraph_map rebuilt from the fixture."""
    tr2data = {int(k): {"entry_id": int(e), "runtime_id": int(r), "timestamp": np.int64(ts), "y": torch.tensor(int(y))}
               for k, e, r, ts, y in zip(z["tr_keys"], z["tr_entry_id"], z["tr_runtime_id"], z["tr_timestamp"],
                                         z["tr_y"])}
    e2r, ptr = {}, z["ent_ptr"]
    for i, e in enumerate(z["ent_keys"].tolist()):
        e2r[e] = dict(zip(z["ent_runtime_id"][ptr[i]:ptr[i + 1]].tolist(), z["ent_prob"][ptr[i]:ptr[i + 1]].tolist()))
    r2g = {}
    for k, rt in enumerate(z["span_keys"].tolist()):
        ms, ei, ea, nd = _fixture_graph(z, "span", k)
        r2g[rt] = {"edge_index": torch.from_numpy(ei), "ms_id": torch.from_numpy(ms).reshape(-1, 1),
                   "occurences": int(z["span_occurences"][k]), "num_nodes": int(z["span_num_nodes"][k]),
                   "node_depth": torch.from_numpy(nd), "edge_attr": torch.from_numpy(ea)}
    return tr2data, e2r, r2g


def _resources(table):
    """A resource row for every (30 s bucket, microservice) of the table, as main() needs."""
    from pert_gnn_kdd23_b200.synthetic import RESOURCE_COLUMNS

    n_ms = int(max(table["um"].max(), table["dm"].max())) + 1
    buckets = np.unique(table["timestamp"] // 30000 * 30000)
    index = [(int(t), m) for t in buckets for m in range(n_ms)]
    vals = np.random.default_rng(0).random((len(index), len(RESOURCE_COLUMNS)))
    return index, vals, n_ms


# ------------------------------------------------------------------------------------------------------------- CPU
def test_oracle_reproduces_reference_main():
    z, table = _golden()
    o = CO.catalogue(table)
    for mine, ref in (("traceid", "tr_keys"), ("entry", "tr_entry_id"), ("runtime_id", "tr_runtime_id"),
                      ("timestamp", "tr_timestamp"), ("y", "tr_y"), ("pat_runtime_id", "span_keys"),
                      ("pat_occurrences", "span_occurences"), ("pat_runtime_id", "pert_keys"),
                      ("pat_occurrences", "pert_occurences"), ("entries", "ent_keys"), ("ent_ptr", "ent_ptr"),
                      ("ent_runtime_id", "ent_runtime_id")):
        assert np.array_equal(o[mine], z[ref]), mine
    assert o["ent_prob"].tobytes() == z["ent_prob"].tobytes()            # float64 bit for bit
    # some pattern's representative (first trace in (entry, traceid) order) is not its smallest traceid
    pat_first = {int(r): int(t) for t, r in zip(z["tr_keys"][::-1], z["tr_runtime_id"][::-1])}
    pat_min = {}
    for t, r in zip(z["tr_keys"].tolist(), z["tr_runtime_id"].tolist()):
        pat_min[r] = min(pat_min.get(r, t), t)
    assert any(pat_first[r] != pat_min[r] for r in pat_min)
    # representatives: the span graphs of the oracle's representative rows are the reference's tensors
    rows, rp = CO.representative_rows(table, o["pat_traceid"])
    keep, new_ptr, roots = pertgraph.clean_span_tables_flat(rows, rp)
    for k in range(len(o["pat_traceid"])):
        kk = keep[new_ptr[k]:new_ptr[k + 1]]
        got = O.span_graph(rows["um"][kk], rows["dm"][kk], rows["interface"][kk], rows["rpctype"][kk], roots[k])
        for g, w in zip(got[:4], _fixture_graph(z, "span", k)):
            assert np.array_equal(np.asarray(g).reshape(np.asarray(w).shape), w), k


def test_fixture_has_the_table_features():
    z, table = _golden()
    tid = table["traceid"]
    assert (np.diff(tid) < 0).any()                                         # traces interleave in file order
    assert len(np.unique(tid)) < tid.max() - tid.min()                      # non-dense ids
    assert (table["um"] == table["dm"]).any()                               # self loops
    _, counts = np.unique(tid, return_counts=True)
    assert (counts == 1).any()                                              # single-row traces
    assert len(z["span_keys"]) >= 15


@pytest.mark.parametrize("case", ["missing", "empty", "dtype", "shape"])
def test_argument_checks_raise_before_launch(case):
    table, _ = make_processed_tables(1, 20)
    if case == "missing":
        del table["interface"]
        err = KeyError
    elif case == "empty":
        table = {k: v[:0] for k, v in table.items()}
        err = ValueError
    elif case == "dtype":
        table["rt"] = table["rt"].astype(np.int32)
        err = TypeError
    else:
        table["um"] = table["um"][:-1]
        err = ValueError
    with pytest.raises(err):
        C.build_catalogue(table, "cuda")


# ------------------------------------------------------------------------------------------------------------- GPU
def _host(cat):
    return {k: getattr(cat, k).cpu().numpy() for k in ("traceid", "entry", "runtime_id", "timestamp", "y",
                                                        "pat_runtime_id", "pat_traceid", "pat_occurrences", "entries",
                                                        "ent_ptr", "ent_runtime_id", "ent_prob")}


def _assert_equal_to_oracle(cat, o):
    h = _host(cat)
    for k, v in o.items():
        if k == "ent_prob":
            assert h[k].tobytes() == v.tobytes(), k
        else:
            assert np.array_equal(h[k], v), k


@pytest.mark.gpu
def test_catalogue_equals_reference_main():
    z, table = _golden()
    cat = C.build_catalogue(table, "cuda")
    assert cat.rekey_rounds == 0
    tr2data, e2r, r2g = cat.to_reference("span")
    ref_tr, ref_e2r, ref_r2g = _fixture_dicts(z)
    assert list(tr2data) == list(ref_tr)
    types = z["tr_types"].tolist()
    for k, v in tr2data.items():
        w = ref_tr[k]
        assert [type(k).__name__] + [type(v[f]).__name__ for f in ("entry_id", "runtime_id", "timestamp", "y")] \
            == types
        assert v["entry_id"] == w["entry_id"] and v["runtime_id"] == w["runtime_id"]
        assert v["timestamp"] == w["timestamp"]
        assert v["y"].dtype == torch.int64 and v["y"].dim() == 0 and int(v["y"]) == int(w["y"])
    assert list(e2r) == list(ref_e2r)
    for e in e2r:
        assert list(e2r[e].items()) == list(ref_e2r[e].items())          # order, keys, float values bit for bit
        assert all(type(p) is float for p in e2r[e].values())
    assert list(r2g) == list(ref_r2g)
    for rt, g in r2g.items():
        w = ref_r2g[rt]
        assert g["occurences"] == w["occurences"] and g["num_nodes"] == w["num_nodes"]
        for f in ("edge_index", "ms_id", "node_depth", "edge_attr"):
            assert g[f].dtype == w[f].dtype and torch.equal(g[f], w[f]), (rt, f)
    # PERT graphs: equal up to the node numbering the reference leaves unspecified
    _, _, p2g = cat.to_reference("pert")
    assert list(p2g) == z["pert_keys"].tolist()
    for k, (rt, g) in enumerate(p2g.items()):
        assert g["occurences"] == int(z["pert_occurences"][k]) and g["num_nodes"] == int(z["pert_num_nodes"][k])
        got = O.canonical_form(g["ms_id"].numpy(), g["edge_index"].numpy(), g["edge_attr"].numpy(),
                               g["node_depth"].numpy())
        assert got == O.canonical_form(*_fixture_graph(z, "pert", k)), rt


def _big_table(seed, long_trace=False):
    table, _ = make_processed_tables(seed, 20000, n_patterns=200, n_entries=24, traceid_base=3 << 31)
    if long_trace:                                                    # one trace of 2,100 rows
        n = 2100
        rng = np.random.default_rng(seed)
        # distinct (um, dm) pairs and rpcids: all 2,100 rows survive the row filters of the graph builders
        extra = {"traceid": np.full(n, 7), "timestamp": 90000 + np.arange(n), "rpcid": np.arange(n),
                 "um": 1 + np.arange(n) % 60, "dm": 1000 + np.arange(n), "interface": rng.integers(0, 16, n),
                 "rpctype": rng.integers(0, 4, n), "rt": rng.integers(1, 50, n), "entryid": np.full(n, 6)}
        extra["um"][0], extra["rt"][0] = 0, 5000
        table = {k: np.concatenate([table[k], extra[k].astype(np.int64)]) for k in table}
    return table


@pytest.mark.gpu
@pytest.mark.parametrize("seed", [1, 2, 3])
def test_catalogue_equals_oracle_at_20k_traces(seed):
    table = _big_table(seed, long_trace=seed == 1)
    assert table["traceid"].max() > 2 ** 31
    cat = C.build_catalogue(table, "cuda")
    _assert_equal_to_oracle(cat, CO.catalogue(table))
    if seed == 1:
        assert int(cat.y.max()) == 5000
        with pytest.raises(pertgraph._lib.PertGnnError):              # graphs keep their 2,048-row limit
            cat.graphs("span")
    # device-resident input gives the same catalogue
    dev = C.build_catalogue({k: torch.from_numpy(v).cuda() for k, v in table.items()}, "cuda")
    _assert_equal_to_oracle(dev, CO.catalogue(table))


@pytest.mark.gpu
@pytest.mark.parametrize("mask", [0x1, 0x7])
def test_forced_hash_collisions_stay_exact(mask):
    table = _big_table(4)
    C._hook = {"hash_mask": mask}
    try:
        cat = C.build_catalogue(table, "cuda")
        hook = C._hook
    finally:
        C._hook = None
    assert hook["rekey_rounds"] > 0 and hook["mismatches"] > 0 and cat.rekey_rounds == hook["rekey_rounds"]
    _assert_equal_to_oracle(cat, CO.catalogue(table))


@pytest.mark.gpu
def test_inconsistent_entry_is_rejected():
    table, _ = make_processed_tables(2, 50)
    i = np.flatnonzero(table["traceid"] == table["traceid"][np.argmax(np.bincount(
        np.unique(table["traceid"], return_inverse=True)[1]))])
    table["entryid"][i[-1]] += 1
    with pytest.raises(pertgraph._lib.PertGnnError, match="entryid"):
        C.build_catalogue(table, "cuda")


@pytest.mark.gpu
def test_store_from_catalogue_equals_dict_store():
    from pert_gnn_kdd23_b200.store import PatternStore

    table, _ = make_processed_tables(6, 600)
    cat = C.build_catalogue(table, "cuda")
    g = cat.graphs("span")
    index, vals, n_ms = _resources(table)
    sa = PatternStore.from_catalogue(cat, g, index, vals, n_ms=n_ms)
    tr2data, e2r, r2g = cat.to_reference("span", graphs=g)
    sb = PatternStore(r2g, e2r, index, vals, tr2data, "cuda", n_ms=n_ms)
    assert len(sa) == len(sb) == len(cat) and sa.trace_keys == sb.trace_keys
    for k in sb.t:
        assert torch.equal(sa.t[k], sb.t[k]), k
    rng = np.random.default_rng(0)
    for ids in ([0], list(range(32)), rng.integers(0, len(cat), 100).tolist(), [len(cat) - 1, 3, 3]):
        ba, bb = sa.assemble(ids), sb.assemble(ids)
        for k in ("x", "edge_index", "edge_attr", "cat_X", "node_depth", "pattern_num_nodes", "rt_probs", "batch",
                  "entry_id", "y", "ptr", "pattern_probs"):
            assert torch.equal(ba[k], bb[k]), k
    sa.check()


@pytest.mark.gpu
def test_span_table_to_train_step():
    """Table -> catalogue -> span graphs -> store -> StoreLoader -> forward + fused_train_step, next to the same
    chain built from the reference's own dicts (the fixture)."""
    import copy

    from pert_gnn_kdd23_b200.model import SAGEDeterministic
    from pert_gnn_kdd23_b200.store import PatternStore, StoreLoader
    from pert_gnn_kdd23_b200.train import FlatParams, FusedAdam, fused_train_step

    z, table = _golden()
    index, vals, n_ms = _resources(table)
    cat = C.build_catalogue(table, "cuda")
    sa = PatternStore.from_catalogue(cat, cat.graphs("span"), index, vals, n_ms=n_ms)
    ref_tr, ref_e2r, ref_r2g = _fixture_dicts(z)
    sb = PatternStore(ref_r2g, ref_e2r, index, vals, ref_tr, "cuda", n_ms=n_ms)
    torch.manual_seed(0)
    model_a = SAGEDeterministic(9, [n_ms], int(table["entryid"].max()), 16, 4, 32, 2, 0.0).cuda()
    model_b = copy.deepcopy(model_a)
    opt_a, opt_b = FusedAdam(FlatParams(model_a), lr=1e-3), FusedAdam(FlatParams(model_b), lr=1e-3)
    ids = list(range(0, len(cat), 3))
    la_, lb_ = StoreLoader(sa, ids, batch_size=25), StoreLoader(sb, ids, batch_size=25)
    for step, (ba, bb) in enumerate(zip(la_, lb_)):
        for k in ("x", "edge_index", "edge_attr", "cat_X", "node_depth", "batch", "ptr", "rt_probs", "y"):
            assert torch.equal(ba[k], bb[k]), k
        if step == 0:
            model_a.eval(), model_b.eval()
            with torch.no_grad():
                args = lambda b: (b.x, b.cat_X, b.edge_index, b.edge_attr, b.pattern_num_nodes, b.rt_probs,  # noqa
                                  b.entry_id, b.batch)
                ya, yb = model_a(*args(ba))[0], model_b(*args(bb))[0]
            assert torch.isfinite(ya).all() and torch.allclose(ya, yb, rtol=1e-5, atol=1e-6)   # pool atomics order
            model_a.train(), model_b.train()
        la, lb = fused_train_step(model_a, opt_a, ba, 0.5), fused_train_step(model_b, opt_b, bb, 0.5)
        assert abs(float(la) - float(lb)) <= 1e-5 * abs(float(lb)), (step, float(la), float(lb))
        if step == 1:
            break
