"""Cost of build_catalogue (pert_gnn_kdd23_b200/catalogue.py, csrc/catalogue.cu) at preprocessing sizes.

Tables of 1e5 and 1e6 traces of 20-40 rows, 1,000 patterns, 64 entries, rows sorted by timestamp (traces interleave).
Reported per size:
  * the whole call from device-resident columns and from host numpy arrays (the latter includes the H2D copy of the
    pageable columns): host clock around calls that end in a device synchronise, median of several calls after warm-up;
  * per-kernel device times (torch.profiler with CUDA activities over one call, in a profiling pass of its own);
  * the summary kernel's algorithmic bytes (perm, row_ptr and the six columns it reads, once, + its five outputs) over
    its time, against the 6,580.9 GB/s the project uses as its HBM peak.  The working set (1e6 traces: ~1.7 GB)
    exceeds the 126 MB L2.
The card's name and power limit are read in the same run.  Usage: python profiles/prof_catalogue.py [out.json]."""
import json
import os
import statistics
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from pert_gnn_kdd23_b200 import catalogue

HBM_PEAK_GBS = 6580.9
REPS = 7


def card():
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit, max_sm_clock"] = q
    except Exception as e:  # noqa: BLE001
        info["power_limit, max_sm_clock"] = f"unavailable: {e!r}"
    return info


def make_table(n_traces, seed=0, n_patterns=1000, n_entries=64, rows=(20, 40), n_ms=4096, n_if=1024):
    """Vectorised table generator (the per-trace loop of synthetic.make_processed_tables is too slow at 1e6)."""
    rng = np.random.default_rng(seed)
    plen = rng.integers(rows[0], rows[1] + 1, n_patterns)
    pptr = np.concatenate([[0], np.cumsum(plen)])
    tot = int(pptr[-1])
    p_um, p_dm, p_if = (rng.integers(1, n_ms, tot), rng.integers(1, n_ms, tot), rng.integers(0, n_if, tot))
    p_um[pptr[:-1]] = 0
    ent_pats = rng.integers(0, n_patterns, (n_entries, 32))
    ent = rng.integers(0, n_entries, n_traces)
    pat = ent_pats[ent, rng.integers(0, 32, n_traces)]
    lens = plen[pat]
    R = int(lens.sum())
    tptr = np.concatenate([[0], np.cumsum(lens)])
    t = np.repeat(np.arange(n_traces), lens)
    k = np.arange(R) - tptr[t]
    src = pptr[pat][t] + k
    t0 = rng.integers(0, 3_600_000, n_traces)
    table = {"traceid": (rng.permutation(n_traces).astype(np.int64) * 7 + (1 << 33))[t],
             "timestamp": t0[t] + 3 * k, "rpcid": k.astype(np.int64), "um": p_um[src], "dm": p_dm[src],
             "interface": p_if[src], "rpctype": rng.integers(0, 8, R), "rt": rng.integers(-500, 500, R),
             "entryid": (ent * 5)[t]}
    table["rt"][tptr[:-1]] = 10_000
    order = np.argsort(table["timestamp"], kind="stable")
    return {c: np.ascontiguousarray(v[order], dtype=np.int64) for c, v in table.items()}, R


def timed(fn):
    fn()
    fn()
    out = []
    for _ in range(REPS):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        out.append(1e3 * (time.perf_counter() - t0))
    return statistics.median(out), min(out), max(out)


def kernel_times(fn):
    from torch.profiler import ProfilerActivity, profile

    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    rows = {}
    for ev in prof.key_averages():
        us = getattr(ev, "device_time_total", None)
        if us is None:
            us = ev.cuda_time_total
        if us > 0:
            rows[ev.key] = {"us": round(us, 1), "calls": ev.count}
    return dict(sorted(rows.items(), key=lambda kv: -kv[1]["us"]))


def main():
    out = {"card": card(), "hbm_peak_gbs": HBM_PEAK_GBS, "sizes": []}
    for n in (100_000, 1_000_000):
        table, R = make_table(n)
        dev_cols = {c: torch.from_numpy(v).cuda() for c, v in table.items()}
        cat = catalogue.build_catalogue(dev_cols, "cuda")
        P, E = cat.num_patterns, int(cat.entries.shape[0])
        d_med, d_min, d_max = timed(lambda: catalogue.build_catalogue(dev_cols, "cuda"))
        h_med, h_min, h_max = timed(lambda: catalogue.build_catalogue(table, "cuda"))
        kt = kernel_times(lambda: catalogue.build_catalogue(dev_cols, "cuda"))
        summ = [v["us"] / v["calls"] for k, v in kt.items() if "k_catalogue_summary" in k]
        summ_bytes = 8 * R + 8 * (n + 1) + 6 * 8 * R + 5 * 8 * n
        rec = {"traces": n, "rows": R, "patterns": P, "entries": E, "rekey_rounds": cat.rekey_rounds,
               "build_from_device_ms": {"median": round(d_med, 3), "min": round(d_min, 3), "max": round(d_max, 3)},
               "build_from_host_ms": {"median": round(h_med, 3), "min": round(h_min, 3), "max": round(h_max, 3)},
               "traces_per_s_from_device": round(n / (d_med * 1e-3)), "kernels_us": kt,
               "summary_bytes": summ_bytes}
        if summ:
            gbs = summ_bytes / (summ[0] * 1e-6) / 1e9
            rec["summary_us"] = round(summ[0], 1)
            rec["summary_gbs"] = round(gbs, 1)
            rec["summary_share_of_hbm_peak"] = round(gbs / HBM_PEAK_GBS, 3)
        out["sizes"].append(rec)
        print(json.dumps({k: v for k, v in rec.items() if k != "kernels_us"}), flush=True)
        del dev_cols, cat
        torch.cuda.empty_cache()
    out["reference_main_cpu_note"] = ("preprocess.py main() on the CPU build host (not a B200, not like-for-like): "
                                      "7.2 s for 20,000 traces of ~5 rows, about 2.8 k traces/s")
    js = json.dumps(out, indent=1)
    print(js)
    if len(sys.argv) > 1:
        with open(sys.argv[1], "w") as f:
            f.write(js + "\n")


if __name__ == "__main__":
    main()
