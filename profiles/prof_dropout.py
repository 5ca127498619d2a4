"""Cost of training-mode dropout (fused into the BatchNorm-apply kernel, csrc/nodeops.cu k_bn_apply<true>).

Three numbers, each variant alternated with the others inside one run (usage on the GPU box:
python profiles/prof_dropout.py [out.json]; without a path the JSON is only printed):
  * ms/step of the graph-replayed train step (train.GraphedTrainStep + fused Adam, resident batches) at cfg2 and cfg3
    for p in {0, 0.1, 0.5} -- CUDA events around blocks of steps, the variants interleaved block by block;
  * the in-step time of the BatchNorm apply of layer 0 (PertProbe kind 6, eagerly issued fused steps), with and
    without dropout;
  * the reference's drop-in loop body (model(...), loss.backward(), torch.optim.Adam, loss.item(); host batches) at
    cfg2 with p = 0.1, through the operator path (use_engine=False: the route a dropout model took before the engine
    ran dropout) and through the engine.
The card's name and power limit are read in the same run."""
import json
import os
import statistics
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

from pert_gnn_kdd23_b200.data import Batch
from pert_gnn_kdd23_b200.engine import PertProbe
from pert_gnn_kdd23_b200.model import SAGEDeterministic
from pert_gnn_kdd23_b200.synthetic import make_data_list, model_args
from pert_gnn_kdd23_b200.train import (FlatParams, FusedAdam, GraphedTrainStep, fused_train_step, model_inputs,
                                       torch_quantile_loss)

PS = (0.0, 0.1, 0.5)
N_ROT = 4


def batches(cfg):
    out = []
    for r in range(N_ROT):
        dl = make_data_list(cfg, seed=1000 + cfg + 131 * r)
        for d in dl:
            d._store.pop("level", None)
            d._store.pop("min_depth", None)
        out.append(Batch.from_data_list(dl))
    return out


def card():
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit, max_sm_clock"] = q
    except Exception as e:  # noqa: BLE001
        info["power_limit, max_sm_clock"] = f"unavailable: {e!r}"
    return info


def make_variant(cfg, p, dev):
    torch.manual_seed(0)                       # same weights for every variant
    model = SAGEDeterministic(*(model_args(cfg)[:-1] + (p,))).to(dev)
    model.train()
    fp = FlatParams(model)
    opt = FusedAdam(fp, lr=3e-4)
    model.engine(fp).seed_dropout(1, 0)
    return {"p": p, "model": model, "opt": opt, "gstep": GraphedTrainStep(model, opt)}


def graph_steps(cfg, dev, blocks=12, k=20):
    dbs = [b.to(dev) for b in batches(cfg)]
    vs = [make_variant(cfg, p, dev) for p in PS]
    for v in vs:
        for i in range(3 * N_ROT):             # eager visit, capture, replays of every batch
            v["gstep"](dbs[i % N_ROT])
    torch.cuda.synchronize()
    times = {v["p"]: [] for v in vs}
    for _ in range(blocks):
        for v in vs:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for i in range(k):
                v["gstep"](dbs[i % N_ROT])
            e1.record()
            e1.synchronize()
            times[v["p"]].append(e0.elapsed_time(e1) / k)
    replays = {v["p"]: v["gstep"].replays for v in vs}
    # in-step BatchNorm-apply time (layer 0), eagerly issued fused steps with the engine's event probe
    bn = {v["p"]: [] for v in vs}
    for r in range(30):
        for v in vs:
            pr = PertProbe.create("bn_apply", 0)
            fused_train_step(v["model"], v["opt"], dbs[r % N_ROT], probe=pr)
            torch.cuda.synchronize()
            bn[v["p"]].append(pr.elapsed_ms())
            pr.destroy()
    N, H = dbs[0].x.size(0), model_args(cfg)[5]
    out = {"nodes": N, "hidden": H, "graphs": dbs[0].num_graphs, "graph_replays": replays}
    base = statistics.median(times[0.0])
    for p in PS:
        med = statistics.median(times[p])
        bmed = statistics.median(bn[p])
        out[f"p={p}"] = {
            "ms_per_step_median": med, "ms_per_step_min": min(times[p]), "ms_per_step_max": max(times[p]),
            "step_overhead_vs_p0_pct": 100.0 * (med / base - 1.0),
            "bn_apply_layer0_us_median": 1e3 * bmed, "bn_apply_layer0_us_min": 1e3 * min(bn[p]),
            # algorithmic bytes of the apply: read x, write y (fp32)
            "bn_apply_GBps_median": 8.0 * N * H / (bmed * 1e-3) / 1e9,
        }
    return out


def dropin(dev, p=0.1, blocks=8, k=15):
    hbs = [b.pin_memory() for b in batches(2)]
    arms = {}
    for name, use_engine in (("operator_path (use_engine=False)", False), ("engine", True)):
        torch.manual_seed(0)
        m = SAGEDeterministic(*(model_args(2)[:-1] + (p,))).to(dev)
        m.use_engine = use_engine
        m.train()
        arms[name] = (m, torch.optim.Adam(m.parameters(), lr=3e-4))

    def step(m, opt, hb):
        data = hb.to(dev, non_blocking=True)
        opt.zero_grad()
        gp, _ = m(*model_inputs(data))
        loss = torch_quantile_loss(data.y.float(), gp.flatten(), 0.5)
        loss.backward()
        opt.step()
        return loss.item()

    for m, opt in arms.values():
        for i in range(8):
            step(m, opt, hbs[i % N_ROT])
    torch.cuda.synchronize()
    times = {n: [] for n in arms}
    for _ in range(blocks):
        for n, (m, opt) in arms.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for i in range(k):
                step(m, opt, hbs[i % N_ROT])
            e1.record()
            e1.synchronize()
            times[n].append(e0.elapsed_time(e1) / k)
    B = hbs[0].num_graphs
    return {n: {"ms_per_step_median": statistics.median(t), "ms_per_step_min": min(t),
                "dags_per_s_median": B / (statistics.median(t) * 1e-3)} for n, t in times.items()}


def main():
    out_path = sys.argv[1] if len(sys.argv) > 1 else None     # without a path the result is only printed
    assert torch.cuda.is_available(), "needs a GPU"
    dev = torch.device("cuda", 0)
    res = {"card": card(), "torch": torch.__version__}
    print(json.dumps({"card": res["card"]}), flush=True)
    for cfg in (2, 3):
        res[f"cfg{cfg}_graph_replay_step"] = graph_steps(cfg, dev)
        print(json.dumps({f"cfg{cfg}": res[f"cfg{cfg}_graph_replay_step"]}, indent=1), flush=True)
    res["cfg2_dropin_loop_p0.1"] = dropin(dev)
    print(json.dumps(res["cfg2_dropin_loop_p0.1"], indent=1), flush=True)
    if out_path:
        os.makedirs(os.path.dirname(out_path) or ".", exist_ok=True)
        with open(out_path, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
