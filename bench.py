#!/usr/bin/env python
"""bench.py -- call-graph DAGs/sec (forward + backward + optimizer step) on B200, per the driver contract.

  python bench.py --gpus N --steps K --warmup W            # this repository's CUDA path
  python bench.py --impl reference --gpus N --steps K ...   # reference-semantics CPU path (oracle) on host cores
  python bench.py ... --dump-outputs DIR                    # also write one step of the timed path as DIR/*.npy

Every timed region of GPU train steps is exactly K steps.  Inputs and initial weights are seeded; --dump-outputs
writes what one step of the timed path computes from the seeded weights, so that two builds run with the same
arguments can be compared output for output.

Workload (BASELINE.json configs[1]): Alibaba-trace-shaped synthetic batch, 256 DAGs x 200 nodes / 600 edges,
64-dim, num_layers=3 (3 TransformerConv + 2 BN), fp32, per GPU (weak scaling for N > 1: every rank trains on
its own 256-graph shard; the gradient mean over the ranks is fused with Adam in one kernel over NVLink peer memory,
train.PeerAdam, with one NCCL all-reduce of the flat gradient as the fallback).

Arms and JSON keys beyond the base contract:
  value         train.GraphedTrainStep on 8 rotating RESIDENT batches: index build + forward + pinball loss +
                backward replayed from one CUDA graph per batch buffer, then the (fused) Adam  [PERT_BENCH_GRAPH=0:
                eager train.fused_train_step]; CUDA events around exactly K steps, max over ranks
  e2e           the same step fed from pinned HOST batches: data.DevicePrefetcher (one H2D copy per step on a side
                stream, one step ahead) + graph replay + Adam + every step's loss read back (train.AsyncLossReader)
  e2e_dropin    the reference's own loop body (pert_gnn.py:219-250) around the drop-in model, unchanged: pinned host
                batch -> .to(device) -> zero_grad -> model.forward -> pinball loss -> backward -> torch Adam -> item()
  kernels       per-kernel in-step times: CUDA events recorded by the engine (PertProbe) around one kernel family per
                step, in eagerly issued train steps run right after the timed region
  roofline      the kernel family with the largest share of the step: algorithmic bytes / its in-step time against
                the measured HBM peak (MEASURED_PEAKS.json); traffic = DRAM bytes from the committed ncu capture
  scatter_max   the BASELINE metric kernel ([E,64] -> [N,64] segment-max): trains of launches over rotating buffers
                larger than L2 (and the single-launch-after-flush time)
  cpu_baseline  the oracle (torch restatement of the reference's PyG 2.4.0 ops) on this box's host cores, thread
                count chosen by a calibration sweep
  clocks        NVML SM clock / throttle reasons sampled inside the timed region
  pert_pipeline (N = 1) span rows -> PERT graphs on the GPU -> resident pattern store -> device-side batch assembly ->
                train step: graph-build rate, DAGs/s from trace ids, DAGs/s of the step on PERT-shaped batches
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

METRIC = "call-graph DAGs/sec (fwd+bwd)"
N_ROT = 8  # distinct resident batches the timed loop rotates over


def _peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured"
    return 6650.0, "fallback"


class ClockSampler:
    """SM clock + throttle reasons sampled DURING the timed region: NVML in a background thread (a query takes well
    under a millisecond, so even a 30 ms region gets samples); falls back to an `nvidia-smi -lms` child process."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None
        self.idx = gpu_index
        self.nv = None
        self._thread = None
        self._stop = False
        self._sm, self._mx, self._reasons = [], [], set()
        try:
            import pynvml

            pynvml.nvmlInit()
            h = None
            try:
                import torch as _t

                uuid = str(_t.cuda.get_device_properties(gpu_index).uuid)
                h = pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + uuid).encode())
            except Exception:
                h = pynvml.nvmlDeviceGetHandleByIndex(gpu_index)
            self.nv = (pynvml, h)
        except Exception:
            self.nv = None

    def _loop(self):
        nv, h = self.nv
        bits = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}
        try:
            mx = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
        except Exception:
            mx = None
        while not self._stop:
            try:
                self._sm.append(float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)))
                if mx is not None:
                    self._mx.append(float(mx))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                for bit, name in bits.items():
                    if r & bit:
                        self._reasons.add(name)
            except Exception:
                pass
            time.sleep(0.003)

    def _stop_nvml(self):
        self._stop = True
        self._thread.join(timeout=2)
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": sorted(self._reasons)}
        if self._sm:
            out["sm_mhz"] = statistics.median(self._sm)
            out["sm_max_mhz"] = max(self._mx) if self._mx else None
            out["samples"] = len(self._sm)
            out["source"] = "nvml"
        return out

    def start(self):
        if self.nv is not None:
            import threading

            self._thread = threading.Thread(target=self._loop, daemon=True)
            self._thread.start()
            return
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), f"--query-gpu={self.Q}",
                                       "--format=csv,noheader,nounits", "-lms", "100"], stdout=self.f,
                                      stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        if self._thread is not None:
            return self._stop_nvml()
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.f.read().strip().splitlines():
            parts = [x.strip() for x in line.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0]))
                mx.append(float(parts[1]))
            except ValueError:
                continue
            for nm, v in zip(names, parts[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        if sm:
            out["sm_mhz"] = statistics.median(sm)
            out["sm_max_mhz"] = max(mx)
            out["samples"] = len(sm)
        out["reasons"] = sorted(reasons)
        try:
            os.unlink(self.f.name)
        except OSError:
            pass
        return out


def make_batches(cfg, rank, count):
    from pert_gnn_kdd23_b200.data import Batch
    from pert_gnn_kdd23_b200.synthetic import make_data_list

    out = []
    for r in range(count):
        dl = make_data_list(cfg, seed=1000 + cfg + 7919 * rank + 131 * r)
        for d in dl:                      # keep exactly the reference's Data schema (pert_gnn.py:163-173) + rt_probs:
            d._store.pop("level", None)   # the generator's test-only ground truth must not inflate the H2D bytes
            d._store.pop("min_depth", None)
        out.append(Batch.from_data_list(dl))
    return out


# ------------------------------------------------------------------------------------------ reference arm
def _calibrate_threads(make_step, cores):
    """The eager CPU path is a chain of small ops: more threads than it can use make it slower (128 threads ran ~10x
    slower than 8-16 on the 128-core box).  Time one small step per candidate thread count and keep the fastest, so
    that the CPU arm is the reference at its best, not at its most oversubscribed."""
    cands = sorted({c for c in (cores, cores // 2, cores // 4, 32, 16, 8, 4) if 1 <= c <= cores}, reverse=True)
    step = make_step()
    best_t, best = cands[-1], float("inf")
    torch.set_num_threads(cands[-1])
    step()                                           # first-touch / allocator warm-up
    for t in cands:
        torch.set_num_threads(t)
        t0 = time.perf_counter()
        step()
        dt = time.perf_counter() - t0
        if dt < best:
            best_t, best = t, dt
    torch.set_num_threads(best_t)
    return best_t


def _sub_batch(cfg, n_graphs, seed_rank=0):
    """A batch of the first n_graphs graphs of the cfg's synthetic data list (bounded CPU sample)."""
    from pert_gnn_kdd23_b200.data import Batch
    from pert_gnn_kdd23_b200.synthetic import make_data_list

    dl = make_data_list(cfg)
    return Batch.from_data_list(dl[:max(1, min(n_graphs, len(dl)))])


def run_reference(args, rank, world):
    """The reference's own CPU implementation of the path.  torch_geometric is not installable here, so this is the
    oracle port (oracle/model_oracle.py: op-for-op torch restatement of PyG 2.4.0 eager) on all host cores."""
    if rank != 0:
        return
    from oracle.model_oracle import OracleSAGEDeterministic, torch_quantile_loss
    from pert_gnn_kdd23_b200.synthetic import CONFIGS, model_args
    from pert_gnn_kdd23_b200.train import model_inputs

    cores_avail = os.cpu_count() or 1
    cfg = args.cfg
    torch.manual_seed(0)
    model = OracleSAGEDeterministic(*model_args(cfg))
    opt = torch.optim.Adam(model.parameters(), lr=3e-4)

    def step(b):
        opt.zero_grad()
        g, _ = model(*model_inputs(b))
        loss = torch_quantile_loss(b.y.float(), g.flatten(), 0.5)
        loss.backward()
        opt.step()
        return float(loss)

    small = _sub_batch(cfg, 32)
    cores = _calibrate_threads(lambda: (lambda: step(small)), cores_avail)
    full = make_batches(cfg, 0, 1)[0]
    B_full = full.num_graphs
    t0 = time.perf_counter()
    step(full)
    t_full = time.perf_counter() - t0
    # bounded sample: the whole --steps/--warmup run has to end within a few minutes on the host cores
    budget = 150.0 / max(1, args.steps + args.warmup)
    B = B_full if t_full <= budget else max(16, int(B_full * budget / t_full))
    batches = [full, make_batches(cfg, 0, 2)[1]] if B == B_full else [_sub_batch(cfg, B), _sub_batch(cfg, B)]
    B = batches[0].num_graphs
    for i in range(args.warmup):
        step(batches[i % 2])
    t0 = time.perf_counter()
    for i in range(args.steps):
        step(batches[i % 2])
    dt = time.perf_counter() - t0
    val = B * args.steps / dt
    c = CONFIGS[cfg]
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": "DAGs/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": _workload_string(cfg, B_full), "global_batch": B_full, "graphs_per_timed_step": B},
        "cpu_baseline": {"value": val, "unit": "DAGs/s", "cores": cores, "kind": "port",
                         "sample": f"{args.steps} train steps (fwd+bwd+Adam), each on {B} of the workload's {B_full} "
                                   f"graphs; {cores} of {cores_avail} host threads (fastest of a calibration sweep); "
                                   "torch restatement of the reference's PyG 2.4.0 eager ops (PyG itself not "
                                   "installable)"},
        "e2e": {"value": val, "unit": "DAGs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------ CUDA arm
def cpu_baseline(cfg, budget_s=25.0):
    from oracle.model_oracle import OracleSAGEDeterministic, torch_quantile_loss
    from pert_gnn_kdd23_b200.synthetic import model_args
    from pert_gnn_kdd23_b200.train import model_inputs

    cores_avail = os.cpu_count() or 1
    torch.manual_seed(0)
    model = OracleSAGEDeterministic(*model_args(cfg))
    opt = torch.optim.Adam(model.parameters(), lr=3e-4)
    b = _sub_batch(cfg, 32)

    def step():
        opt.zero_grad()
        g, _ = model(*model_inputs(b))
        loss = torch_quantile_loss(b.y.float(), g.flatten(), 0.5)
        loss.backward()
        opt.step()
        return float(loss)

    cores = _calibrate_threads(lambda: step, cores_avail)
    b = make_batches(cfg, 0, 1)[0]
    B = b.num_graphs
    step()
    times = []
    t_start = time.perf_counter()
    while len(times) < 10 and (time.perf_counter() - t_start) < budget_s:
        t0 = time.perf_counter()
        step()
        times.append(time.perf_counter() - t0)
    med = statistics.median(times)
    return {"value": B / med, "unit": "DAGs/s", "cores": cores, "kind": "port",
            "sample": f"{len(times)} full train steps (fwd+bwd+Adam) of the same {B}-graph cfg{cfg} batch, median; "
                      f"{cores} of {cores_avail} host threads (fastest of a calibration sweep); "
                      "oracle = torch restatement of the reference's PyG 2.4.0 eager ops"}


_BENCH_CFG = 2


def ncu_traffic(kernel):
    """DRAM bytes per launch (read + write) of a kernel family from the committed ncu --set full capture
    (profiles/r1_traffic.json, cfg2 shapes only); None when there is no capture for it."""
    if _BENCH_CFG != 2:
        return None
    try:
        with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "profiles", "r2_traffic.json")) as f:
            return json.load(f).get(kernel)
    except (OSError, ValueError):
        return None


def scatter_max_bench(batch_dev, H, peak_gbs, iters=40):
    """BASELINE metric kernel: segment-max of msg[E,H] (CSR order) -> out[N,H].

    Two protocols, both with cold inputs: (a) "single": one launch between two events after a 512 MB L2 flush
    (includes the ~3-5 us launch / event gap of a lone short kernel); (b) "train": TRAIN back-to-back launches over
    ROT distinct message/output buffers whose total footprint exceeds L2 (inputs larger than L2, no flush), one
    event pair around the train, divided by TRAIN -- the per-launch duration once the launch gap is amortised,
    which is what the ncu gpu__time_duration of the same kernel shows.  `frac` is quoted from (b)."""
    from pert_gnn_kdd23_b200 import _lib
    from pert_gnn_kdd23_b200.index import build_index

    N, E = batch_dev.x.size(0), batch_dev.edge_index.size(1)
    gi = build_index(batch_dev.edge_index, N)
    bytes_alg = 4 * E * H + 4 * (N + 1) + 4 * N * H
    ROT = max(4, int(3 * (160 << 20) // max(bytes_alg, 1)) + 1)     # >= 3 x 160 MB of distinct data in rotation
    TRAIN = 2 * ROT
    msgs = [torch.randn(E, H, device="cuda") for _ in range(ROT)]
    outs = [torch.empty(N, H, device="cuda") for _ in range(ROT)]
    flush = torch.empty(512 << 20, dtype=torch.uint8, device="cuda")
    st = torch.cuda.current_stream()

    def launch(i):
        _lib.call("pert_segment_reduce_fwd", msgs[i % ROT].data_ptr(), gi.rowptr.data_ptr(), None,
                  outs[i % ROT].data_ptr(), N, H, 1, st.cuda_stream)

    single = []
    for i in range(iters + 5):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(st)
        launch(i)
        e1.record(st)
        e1.synchronize()
        if i >= 5:
            single.append(e0.elapsed_time(e1) * 1e-3)
    train = []
    for rep in range(12):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(st)
        for i in range(TRAIN):
            launch(i)
        e1.record(st)
        e1.synchronize()
        if rep >= 2:
            train.append(e0.elapsed_time(e1) * 1e-3 / TRAIN)
    t_single, t_train = statistics.median(single), statistics.median(train)
    ach = bytes_alg / t_train / 1e9
    return {"kernel": "k_segreduce_stream<max> [E,H]->[N,H] (TMA bulk + mbarrier pipeline)", "bound": "hbm",
            "achieved": ach, "peak": peak_gbs, "unit": "GB/s", "frac": ach / peak_gbs, "traffic": ncu_traffic("scatter_max"),
            "algorithmic_bytes": bytes_alg, "us_per_launch": t_train * 1e6,
            "protocol": f"{TRAIN} back-to-back launches over {ROT} distinct msg/out buffer pairs "
                        f"({ROT * bytes_alg >> 20} MB > L2), event pair around the train, median of 10",
            "us_single_launch_after_l2_flush": t_single * 1e6,
            "achieved_single_launch": bytes_alg / t_single / 1e9, "shape": {"E": E, "N": N, "H": H}}


def _workload_string(cfg, B):
    """config.workload -- the SAME string in both arms (the driver compares them)."""
    from pert_gnn_kdd23_b200.synthetic import CONFIGS

    c = CONFIGS[cfg]
    nodes = c["nodes"] if c["nodes"] is not None else "20-500 (power law)"
    edges = c["edges"] if c["edges"] is not None else "3x nodes"
    return (f"cfg{cfg}: {B} DAGs x {nodes} nodes/{edges} edges per GPU, {c['hidden']}-dim, "
            f"num_layers={c['num_layers']}, fwd+bwd+Adam")


def timed_steps(run_block, K, barrier, world, dev):
    """Seconds taken by EXACTLY K steps: barrier + synchronize on both sides, a CUDA event pair around the K steps, max
    over ranks."""
    import torch.distributed as dist

    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    run_block(K)
    e1.record()
    barrier()
    secs = e0.elapsed_time(e1) * 1e-3
    if world > 1:
        t = torch.tensor([secs], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        secs = float(t)
    return secs


def dump_step(out_dir, step, opt, fp, model, init, batch):
    """Runs ``step``, one step of the timed path (graph replay of forward + backward, then Adam), on ``batch`` from
    the seeded initial state ``init`` -- parameters, BatchNorm buffers, fresh Adam moments -- and, when ``out_dir`` is
    set, writes what it hands its caller as float .npy files: the loss, the flat gradient buffer it computed, the flat
    parameter buffer after the Adam update (the engine's own layout, one 256-byte-aligned slot per parameter) and the
    BatchNorm buffers.  Collective for N > 1; only rank 0 passes ``out_dir``.
    A step from fixed inputs is what can be compared: the kernels accumulate some sums with float atomics, so two runs
    differ in the last bits of every step, and over many steps Adam (whose first updates are ~lr * sign(gradient))
    and the BatchNorm ReLUs amplify that -- two identical trainings on one B200 differed in their gradients by 4e-6
    after one step, 1e-3 after two and 5e-2 after fifteen.  Two runs of this dump (cfg2, one B200) agreed on the loss
    exactly, on the gradients to 6e-8 of the largest and on the parameters to 4e-5 of the largest; that last figure
    is the lin_skip.bias in front of each BatchNorm, whose gradient is zero in exact arithmetic (rounding noise of
    1e-8) and which Adam's first update moves by up to lr regardless; every other parameter agreed within 2e-6."""
    import numpy as np

    with torch.no_grad():
        fp.flat.copy_(init["flat"])
        opt.m.zero_()
        opt.v.zero_()
        opt.t = 0
        for n, b in model.named_buffers():
            b.copy_(init[n])
    loss = step(batch)
    torch.cuda.synchronize()
    if out_dir is None:
        return
    arrays = {"loss": loss, "grads": fp.grad, "params": fp.flat}
    arrays.update({f"buffer.{n}": b for n, b in model.named_buffers()})
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        a = t.detach().cpu().numpy()
        np.save(os.path.join(out_dir, name + ".npy"), a.astype(np.float32 if a.dtype == np.float32 else np.float64))


def first_step_parity(model, batch_host, dev, tau=0.5):
    """The step's first forward against the oracle bench.py already ships for its CPU arm: same weights, same batch,
    training-mode BatchNorm; asserts predictions (element-wise) and loss within 1e-4 before anything is timed."""
    import copy

    from oracle.model_oracle import OracleSAGEDeterministic, torch_quantile_loss
    from pert_gnn_kdd23_b200.synthetic import model_args
    from pert_gnn_kdd23_b200.train import model_inputs

    m = copy.deepcopy(model)
    oracle = OracleSAGEDeterministic(*model_args(_BENCH_CFG))
    oracle.load_state_dict({k: v.detach().cpu() for k, v in m.state_dict().items()})
    oracle.train()
    m.train()
    with torch.no_grad():
        go, _ = oracle(*model_inputs(batch_host))
        gc, _ = m(*model_inputs(batch_host.to(dev)))
    lo = float(torch_quantile_loss(batch_host.y.float(), go.flatten(), tau))
    lc = float(torch_quantile_loss(batch_host.y.float().to(dev), gc.flatten(), tau))
    d = (gc.cpu().double() - go.double()).abs()
    rms = go.double().pow(2).mean().sqrt()
    elem = float((d / (go.double().abs() + rms)).max())
    out = {"loss_cuda": lc, "loss_oracle": lo, "loss_rel_err": abs(lc - lo) / max(abs(lo), 1e-30),
           "pred_elementwise_rel_err": elem, "bar": 1e-4}
    assert out["loss_rel_err"] <= 1e-4 and elem <= 1e-4, f"first-step parity vs the oracle failed: {out}"
    return out


def run_b200(args, rank, world, local_rank):
    import torch.distributed as dist

    from pert_gnn_kdd23_b200 import ops
    from pert_gnn_kdd23_b200.data import DevicePrefetcher
    from pert_gnn_kdd23_b200.engine import PertProbe
    from pert_gnn_kdd23_b200.model import SAGEDeterministic
    from pert_gnn_kdd23_b200.synthetic import CONFIGS, model_args
    from pert_gnn_kdd23_b200.train import (AsyncLossReader, DataParallel, FlatParams, FusedAdam, GraphedTrainStep,
                                           fused_train_step, model_inputs, torch_quantile_loss)

    train_step = fused_train_step

    assert torch.cuda.is_available(), "bench.py (CUDA arm) needs a GPU; there is no CPU fallback"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    cfg = args.cfg
    c = CONFIGS[cfg]
    H = c["hidden"]
    peak, peak_kind = _peaks()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def make_optimizer(fp):
        # N > 1: the gradient all-reduce is fused with Adam in one kernel over NVLink peer memory (train.PeerAdam);
        # PERT_BENCH_PEER=0 (or a failed IPC setup) falls back to one NCCL all_reduce of the flat gradient + fused Adam
        opt, sync = None, "single GPU: fused Adam"
        if world > 1 and os.environ.get("PERT_BENCH_PEER", "1") != "0":
            from pert_gnn_kdd23_b200.train import PeerAdam

            ok = torch.ones(1, device=dev)
            try:
                opt = PeerAdam(fp, lr=3e-4)
                sync = "PeerAdam: gradient all-reduce fused with Adam in one kernel over NVLink peer memory (no NCCL)"
            except Exception:  # noqa: BLE001
                ok.zero_()
            dist.all_reduce(ok, op=dist.ReduceOp.MIN)
            if float(ok) == 0.0:
                opt = None
        if opt is None:
            opt = FusedAdam(fp, lr=3e-4)
            if world > 1:
                sync = "NCCL all_reduce of the flat gradient + fused Adam"
        return opt, sync

    host_batches = [b.pin_memory() for b in make_batches(cfg, rank, N_ROT)]
    dev_batches = [b.to(dev) for b in host_batches]
    B = host_batches[0].num_graphs
    Nn, Ee = host_batches[0].x.size(0), host_batches[0].edge_index.size(1)
    h2d = host_batches[0].h2d_bytes

    torch.manual_seed(0)
    model = SAGEDeterministic(*model_args(cfg)).to(dev)
    parity = None
    if rank == 0 and not args.no_parity_check:
        parity = first_step_parity(model, make_batches(cfg, rank, 1)[0], dev)
    fp = FlatParams(model)
    opt, grad_sync = make_optimizer(fp)
    dp = DataParallel(fp) if world > 1 else None
    init = {"flat": fp.flat.clone(), **{n: b.clone() for n, b in model.named_buffers()}}

    # ---- kernel-only arm: inputs resident in HBM -------------------------------------------------
    # The step is replayed from a CUDA graph per resident batch (train.GraphedTrainStep: index build + forward +
    # loss + backward in one cudaGraphLaunch, then the eager all-reduce / Adam); PERT_BENCH_GRAPH=0 times the eager
    # fused step instead.  A key is captured on its second visit, so the warm-up visits every batch at least twice.
    use_graph = os.environ.get("PERT_BENCH_GRAPH", "1") != "0"
    gstep = GraphedTrainStep(model, opt, 0.5, dp)

    def stepper(d):
        return gstep(d) if use_graph else train_step(model, opt, d, 0.5, dp)

    state = {"i": 0, "loss": None}

    def resident_block(k):
        for _ in range(k):
            state["loss"] = stepper(dev_batches[state["i"] % N_ROT])
            state["i"] += 1

    resident_block(max(args.warmup, 2 * N_ROT))
    barrier()
    if hasattr(opt, "phase_times_us"):
        opt.phase_times_us(reset=True)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    l0 = ops.LAUNCHES["n"]
    s0 = state["i"]
    t_wall = time.perf_counter()
    secs = timed_steps(resident_block, args.steps, barrier, world, dev)
    t_wall = time.perf_counter() - t_wall
    launches_per_step = (ops.LAUNCHES["n"] - l0) / max(1, state["i"] - s0)
    clocks = sampler.stop() if rank == 0 else None
    peer_phases = opt.phase_times_us(reset=True) if hasattr(opt, "phase_times_us") and world > 1 else None
    loss = float(state["loss"])          # read now: the dumped step below reuses the graph's loss buffer
    last_batch = dev_batches[(state["i"] - 1) % N_ROT]
    value = world * B * args.steps / secs

    # ---- in-step kernel durations: the engine records a caller-created CUDA event pair around ONE kernel family of
    # the middle layer per step (include/pertgnn.h PertProbe), in eagerly issued steps right after the timed region
    # (events inside a replayed graph cannot be timed)
    n_convs = len(model.convs)
    fams = ["tconv_bwd", "tconv_fwd", "gemm_fwd", "gemm_wgrad", "gemm_dgrad"]
    n_probe = max(2 * len(fams), min(args.steps, 40))
    probes = [PertProbe.create(fams[i % len(fams)], min(1, n_convs - 1)) for i in range(n_probe)]
    for i in range(n_probe):
        train_step(model, opt, dev_batches[i % N_ROT], 0.5, dp, probe=probes[i])
    barrier()
    kern = {}
    for i, pr in enumerate(probes):
        kern.setdefault(fams[i % len(fams)], []).append(pr.elapsed_ms())
        pr.destroy()

    # ---- end-to-end arm: the reference's loop body with host buffers ------------------------------
    model2 = SAGEDeterministic(*model_args(cfg)).to(dev)
    model2.load_state_dict(model.state_dict())
    opt2 = torch.optim.Adam(model2.parameters(), lr=3e-4)
    dp2 = DataParallel(FlatParams(model2, bind_grads=False)) if world > 1 else None

    def e2e_step(hb):
        data = hb.to(dev, non_blocking=True)
        opt2.zero_grad()
        gp, _ = model2(*model_inputs(data))
        l = torch_quantile_loss(data.y.float(), gp.flatten(), 0.5)
        l.backward()
        if dp2 is not None:
            dp2.all_reduce_module_grads(model2)       # ONE all-reduce of the engine's flat gradient buffer
        opt2.step()
        return l.item()                       # D2H read of the step's result, like pert_gnn.py:248

    st2 = {"i": 0}

    def dropin_block(k):
        for _ in range(k):
            e2e_step(host_batches[st2["i"] % N_ROT])
            st2["i"] += 1

    dropin_block(args.warmup)
    secs2 = timed_steps(dropin_block, args.steps, barrier, world, dev)
    e2e_val = world * B * args.steps / secs2

    # ---- end-to-end through the fused public API: pinned host batch -> device -> graph-replayed step -> loss read-back
    # every step's inputs cross PCIe inside the timed region (one pinned slab -> one H2D copy per step), issued on a
    # side stream while the previous batch trains (data.DevicePrefetcher); every step's loss is read back (4 B D2H into
    # pinned memory + event, train.AsyncLossReader), consumed one step later so the GPU never idles on the read-back
    pf_ring = DevicePrefetcher([], dev)       # ONE prefetcher: its 3 device slabs (= 3 graph keys) persist across runs
    reader = AsyncLossReader(dev)
    st3 = {"i": 0}

    def fused_block(nsteps):
        total = 0.0
        pf_ring.batches = [host_batches[(st3["i"] + j) % N_ROT] for j in range(nsteps)]
        st3["i"] += nsteps
        for data in pf_ring:
            v = reader.push(stepper(data))
            if v is not None:
                total += v
        v = reader.flush()
        return total + (v if v is not None else 0.0)

    fused_block(max(args.warmup, 9))
    secs3 = timed_steps(fused_block, args.steps, barrier, world, dev)
    e2e_fused_val = world * B * args.steps / secs3

    # ---- BASELINE.json configs[3] (4096 graphs over 8 GPUs = 512 graphs / GPU, 128-dim, 3 layers) beside the headline
    cfg4 = run_cfg4_block(args, rank, world, dev, barrier, make_optimizer) if (args.cfg == 2 and not args.no_cfg4) else None
    cfg2j = run_jitter_block(args, rank, world, dev, barrier, make_optimizer) if (args.cfg == 2 and not args.no_cfg4) else None
    pert_pipe = None
    if args.cfg == 2 and not args.no_cfg4 and world == 1:
        try:
            pert_pipe = run_pert_pipeline_block(args, dev, barrier)
        except Exception as e:  # noqa: BLE001 -- a supplementary block must not take the headline line down
            pert_pipe = {"error": repr(e)[:300]}

    if args.dump_outputs:
        dump_step(args.dump_outputs if rank == 0 else None, stepper, opt, fp, model, init, last_batch)
    if hasattr(opt, "check"):
        opt.check()
    if rank != 0:
        return
    # ---- roofline of the dominant instrumented kernel (bytes model: DESIGN.md section 4) -----------
    Kin = H   # middle layer: K = H
    alg = {   # algorithmic bytes per launch (DESIGN.md section 3)
        "tconv_fwd": 16 * Nn * H + 12 * Ee + 4 * (Nn + 1) + 4 * Ee,
        "tconv_bwd": 2 * (16 * Nn * H + 12 * Ee + 4 * (Nn + 1) + 8 * Ee),
        "gemm_fwd": 4 * Nn * Kin + 16 * Nn * H, "gemm_dgrad": 4 * Nn * Kin + 16 * Nn * H,
        "gemm_wgrad": 4 * Nn * Kin + 16 * Nn * H,
    }
    names = {"tconv_fwd": "fused conv forward (csrc/tconv_tile.cu)",
             "tconv_bwd": "fused conv backward: target pass + source pass (csrc/tconv_tile.cu, 2 launches)",
             "gemm_fwd": "k_gemm_nt_tma (node linears, tcgen05 3xTF32, TMA-tiled)",
             "gemm_dgrad": "k_gemm_nt_tma (data gradient)", "gemm_wgrad": "k_gemm_tn_tma (weight + bias gradient)"}
    kernels = {}
    for name, ts in kern.items():
        ts = [t for t in ts if t == t]
        if not ts:
            continue
        med = statistics.median(ts)
        kernels[name] = {"us_per_launch": 1e3 * med, "launches_per_step": n_convs,
                         "ms_per_step": med * n_convs, "samples": len(ts),
                         "GBs": alg[name] / (med * 1e-3) / 1e9, "frac_of_hbm_peak": alg[name] / (med * 1e-3) / 1e9 / peak}
    roof = None
    if kernels:
        top = max(kernels, key=lambda k: kernels[k]["ms_per_step"])
        ach = kernels[top]["GBs"]
        roof = {"kernel": names[top], "bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s",
                "frac": ach / peak, "traffic": ncu_traffic(top),
                "traffic_source": "committed ncu --set full capture of this command (profiles/r2_traffic.json), "
                                  "NOT measured in this run; below the algorithmic bytes when outputs stay dirty in L2",
                "peak_source": peak_kind, "algorithmic_bytes": alg[top],
                "us_per_launch": kernels[top]["us_per_launch"],
                "share_of_step": kernels[top]["ms_per_step"] / (1e3 * secs / args.steps),
                "how": "CUDA event pair recorded by the engine around the launch(es) inside eagerly issued train "
                       "steps run right after the timed region (middle layer), median over the sampled steps"}
    smx = scatter_max_bench(dev_batches[0], H, peak)
    base = cpu_baseline(cfg) if (world == 1 and not args.no_cpu_baseline) else None
    line = {
        "metric": METRIC, "value": value, "unit": "DAGs/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * secs / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": _workload_string(cfg, B),
                   "global_batch": world * B, "nodes_per_gpu": Nn, "edges_per_gpu": Ee,
                   "convs": n_convs, "parallelism": f"dp{world}", "grad_sync": grad_sync,
                   "step_issue": ("CUDA-graph replay per batch buffer (index build + forward + loss + backward), eager "
                                  f"all-reduce + Adam; {gstep.replays} replays, capture_error={gstep.capture_error}")
                   if use_graph else "eager fused_train_step (5 C calls per step)",
                   "timing": f"exactly {args.steps} steps bracketed by barrier + synchronize and a CUDA event pair, "
                             f"max over ranks (timed region {secs:.3f} s)",
                   "l2": f"rotating {N_ROT} distinct resident batches; ~{(n_convs * 8 * Nn * H * 4) >> 20} MB of "
                         "activations written+read per step (> 126 MB L2 for cfg2+): no explicit flush in the step "
                         "loop; scatter_max is timed with an explicit 512 MB L2 flush"},
        "roofline": roof, "scatter_max": smx, "kernels": kernels, "cpu_baseline": base,
        "e2e_dropin": {"value": e2e_val, "unit": "DAGs/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4,
                "ms_per_step": 1e3 * secs2 / args.steps,
                "path": "pert_gnn.py loop body: Batch.to(device) from pinned host slab, zero_grad, forward, pinball "
                        "loss, backward, torch.optim.Adam.step, float(loss)"},
        "e2e": {"value": e2e_fused_val, "unit": "DAGs/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4,
                      "ms_per_step": 1e3 * secs3 / args.steps,
                      "path": "data.DevicePrefetcher (pinned slab -> one H2D per step on a side stream, overlapped with "
                              "the previous step) + train.GraphedTrainStep (graph replay of index build, engine fwd, "
                              "pinball kernel, engine bwd; eager fused Adam) + the loss of EVERY step read back "
                              "(train.AsyncLossReader: 4-byte D2H + event behind each step, consumed one step later)"},
        "gpu_launches": int(round(launches_per_step * args.steps)),
        "gpu_launches_how": "kernels launched per step through the C-ABI (counted at every binding call: the engine's "
                            "launch list mirrored from csrc/engine.cu + index build + loss + Adam) x steps of one block; "
                            "cross-check: profiles/r2_launches_step.csv (ncu launch list of the same command)",
        "wall_s": t_wall, "clocks": clocks, "final_loss": float(loss), "parity_first_step": parity,
        "peer": peer_phases, "cfg4": cfg4, "cfg2_jittered": cfg2j, "pert_pipeline": pert_pipe,
    }
    print(json.dumps(line), flush=True)


def run_extra_block(args, rank, world, dev, barrier, make_optimizer, cfg, per_gpu, jitter, workload):
    """A second workload measured beside the headline (same step machinery: resident batches, graph replay, fused
    Adam / PeerAdam): every rank trains on its own `per_gpu`-graph batches of config `cfg`."""
    from pert_gnn_kdd23_b200.data import Batch
    from pert_gnn_kdd23_b200.model import SAGEDeterministic
    from pert_gnn_kdd23_b200.synthetic import make_data_list, model_args
    from pert_gnn_kdd23_b200.train import DataParallel, FlatParams, GraphedTrainStep

    n_rot = 3
    batches = []
    for r in range(n_rot):
        dl = make_data_list(cfg, num_graphs=per_gpu, seed=1000 + cfg + 7919 * rank + 131 * r, jitter=jitter)
        for d in dl:
            d._store.pop("level", None)
            d._store.pop("min_depth", None)
        batches.append(Batch.from_data_list(dl).pin_memory().to(dev))
    torch.manual_seed(0)
    model = SAGEDeterministic(*model_args(cfg)).to(dev)
    fp = FlatParams(model)
    opt, sync = make_optimizer(fp)
    dp = DataParallel(fp) if world > 1 else None
    gstep = GraphedTrainStep(model, opt, 0.5, dp)
    st = {"i": 0}

    def block(k):
        for _ in range(k):
            gstep(batches[st["i"] % n_rot])
            st["i"] += 1

    block(max(3, 2 * n_rot + 1))
    barrier()
    if hasattr(opt, "phase_times_us"):
        opt.phase_times_us(reset=True)
    K = args.steps
    secs = timed_steps(block, K, barrier, world, dev)
    phases = opt.phase_times_us(reset=True) if hasattr(opt, "phase_times_us") and world > 1 else None
    if hasattr(opt, "check"):
        opt.check()
    if hasattr(opt, "close"):
        opt.close()
    Nn, Ee = batches[0].x.size(0), batches[0].edge_index.size(1)
    return {"workload": workload, "value": world * per_gpu * K / secs, "unit": "DAGs/s", "global_batch": world * per_gpu,
            "ms_per_step": 1e3 * secs / K, "steps": K, "nodes_per_gpu": Nn,
            "edges_per_gpu": Ee, "grad_sync": sync, "peer": phases, "replays": gstep.replays,
            "capture_error": gstep.capture_error}


def run_cfg4_block(args, rank, world, dev, barrier, make_optimizer):
    """BASELINE.json configs[3]: the 4096-graph batch sharded data-parallel over 8 GPUs = 512 graphs per GPU, 128-dim,
    3 layers, gradient all-reduce fused with Adam.  Measured beside the cfg2 headline (which stays the weak-scaling
    curve): every rank trains on its own 512-graph shard; at N < 8 it is the same per-GPU shard on fewer GPUs."""
    return run_extra_block(args, rank, world, dev, barrier, make_optimizer, 4, 512, 0.0,
                           "BASELINE configs[3] shard: 512 DAGs x 200 nodes/600 edges per GPU (4096 over 8 GPUs), "
                           "128-dim, num_layers=3, fwd+bwd+Adam, resident batches, graph replay")


def run_jitter_block(args, rank, world, dev, barrier, make_optimizer):
    """cfg2 with graph sizes 200 +- 20 % nodes (edges scale along): BASELINE says "~200 nodes / ~600 edges"; the headline
    batch is exactly uniform, real batches are not (graph-aligned tiles, csrc/tconv_tile.cu:k_build_tiles)."""
    return run_extra_block(args, rank, world, dev, barrier, make_optimizer, 2, 256, 0.2,
                           "cfg2j: 256 DAGs x 200 +- 20 % nodes (3 edges per node) per GPU, 64-dim, num_layers=3, "
                           "fwd+bwd+Adam, resident batches, graph replay")


def run_pert_pipeline_block(args, dev, barrier):
    """SURVEY rows N2 + N1 + N4 in front of the train step, all on the GPU: span rows -> PERT graphs
    (pertgraph.build_pert_graphs) -> resident pattern store -> batches of 256 traces assembled on the device
    (store.StoreLoader: sample assembly incl. the (timestamp, ms) feature join + collation) -> fused train step.
    `from_trace_ids`: every step assembles its batch from 256 trace ids (2 KB of H2D) and trains on it;
    `resident_graph_replay`: the train step alone on assembled PERT-shaped batches (comparable with `value`)."""
    from pert_gnn_kdd23_b200.model import SAGEDeterministic
    from pert_gnn_kdd23_b200.store import PatternStore, StoreLoader
    from pert_gnn_kdd23_b200.synthetic import make_pert_artifacts, model_args
    from pert_gnn_kdd23_b200.train import FlatParams, FusedAdam, GraphedTrainStep, fused_train_step

    art, info = make_pert_artifacts(seed=3, n_patterns=256, n_entries=64, n_traces=4096, device=dev)
    art2, info2 = make_pert_artifacts(seed=3, n_patterns=256, n_entries=64, n_traces=4096, device=dev)   # warm timing
    store = PatternStore.from_artifacts(art, dev)
    B = 256
    ids = list(range(len(store)))
    torch.manual_seed(0)
    model = SAGEDeterministic(*model_args(2)).to(dev)
    opt = FusedAdam(FlatParams(model), lr=1e-3)
    loader = StoreLoader(store, ids, batch_size=B)
    nb = len(loader)

    def epoch_block(k):                         # k steps, each: assemble 256 traces on the device + train
        done = 0
        while done < k:
            for batch in loader:
                fused_train_step(model, opt, batch, 0.5)
                done += 1
                if done == k:
                    break

    epoch_block(5)
    barrier()
    K = args.steps
    secs = timed_steps(epoch_block, K, barrier, 1, dev)
    store.check()
    res = [store.assemble(ids[i * B:(i + 1) * B]) for i in range(3)]
    gstep = GraphedTrainStep(model, opt, 0.5, None)
    st = {"i": 0}

    def block(k):
        for _ in range(k):
            gstep(res[st["i"] % 3])
            st["i"] += 1

    block(7)
    barrier()
    secs2 = timed_steps(block, K, barrier, 1, dev)
    Nn, Ee = int(res[0].x.size(0)), int(res[0].edge_index.size(1))
    return {"workload": f"PERT-exact synthetic: {B} traces per step, one PERT graph each (60-72 calls: nodes = 2 calls + "
                        "distinct ms, edges = 4 calls), 64-dim, num_layers=3, fwd+bwd+Adam",
            "graph_build": {"patterns": info2["patterns"], "span_rows": info2["span_rows"], "pert_nodes": info2["nodes"],
                            "pert_edges": info2["edges"], "ms": 1e3 * info2["build_s"],
                            "patterns_per_s": info2["patterns"] / info2["build_s"],
                            "what": "host span rows -> H2D -> count + build kernels -> level index -> node_depth"},
            "from_trace_ids": {"value": B * K / secs, "unit": "DAGs/s", "ms_per_step": 1e3 * secs / K,
                               "h2d_bytes_per_step": 8 * B,
                               "what": "device-side sample assembly + collation from the resident store, then the eager "
                                       "fused train step"},
            "resident_graph_replay": {"value": B * K / secs2, "unit": "DAGs/s", "ms_per_step": 1e3 * secs2 / K,
                                      "replays": gstep.replays,
                                      "capture_error": gstep.capture_error},
            "nodes_per_batch": Nn, "edges_per_batch": Ee, "store_resident_bytes": store.resident_bytes}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--cfg", type=int, default=2)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-parity-check", action="store_true")
    ap.add_argument("--no-cfg4", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what one step of the timed path computes from the seeded "
                         "weights on the last timed batch (loss, gradients, updated parameters) to DIR")
    args = ap.parse_args()
    global _BENCH_CFG
    _BENCH_CFG = args.cfg
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    args.warmup = max(args.warmup, 3)
    run_b200(args, rank, world, local_rank)
    if world > 1:
        import torch.distributed as dist

        dist.destroy_process_group()


if __name__ == "__main__":
    main()
