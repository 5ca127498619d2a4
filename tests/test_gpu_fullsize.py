"""-m gpu parity tests AT THE SIZES BASELINE.json NAMES, so that the kernels bench.py times are the kernels checked:
  * k_segreduce_stream (the BASELINE metric kernel; only dispatched for N >= 4096) at cfg2's real shape and around it;
  * the tcgen05 / TMA GEMMs (NT forward into planes, data gradient out of blocked planes, TN weight gradient with the
    fused bias column sums; only dispatched for M >= 1024 / R >= 4096) at M, R in {4096, 51200, 102400} x H in {64,128};
  * the whole model (outputs, loss, every gradient, BN statistics) on the FULL cfg2 / cfg3 / cfg5 batches and a cfg4
    per-GPU shard, against the CPU oracle.
Bars: max bit-exact; sums / model 1e-4 element-wise (tests/helpers.py:elem_err); GEMMs 2e-6 (K <= 144) .. 8e-6
(K = 512) norm-wise and 5x that element-wise, against fp64."""
import math

import pytest
import torch

from oracle import model_oracle
from tests.helpers import (RTOL, assert_close, assert_grads_close, forward_args, make_batch, make_models)

pytestmark = pytest.mark.gpu


# ------------------------------------------------------------------ the BASELINE metric kernel at its real shapes
def _seg_case(N, H, degs, op, seed=0):
    from pert_gnn_kdd23_b200 import ops

    g = torch.Generator().manual_seed(seed)
    rowptr = torch.zeros(N + 1, dtype=torch.int64)
    rowptr[1:] = torch.cumsum(degs, 0)
    E = int(rowptr[-1])
    msg = torch.randn(E, H, generator=g)
    dst = torch.repeat_interleave(torch.arange(N), degs)
    ref = model_oracle.scatter(msg, dst, N, op)
    out = ops.segment_reduce(msg.cuda(), rowptr.to(torch.int32).cuda(), None, op)
    if op == "max":
        assert torch.equal(out.cpu(), ref), f"segment max differs N={N} H={H}"
    else:
        assert_close(out, ref, what=f"segsum N={N} H={H}")


@pytest.mark.parametrize("H", [32, 64, 128])
@pytest.mark.parametrize("op", ["max", "sum"])
def test_segreduce_stream_cfg2_shape(H, op):
    """cfg2's real CSR (E=153,600 / N=51,200) -> k_segreduce_stream (N >= 4096, H in {32,64,128})."""
    from pert_gnn_kdd23_b200 import ops
    from pert_gnn_kdd23_b200.index import build_index

    b = make_batch(2)
    N, E = b.x.size(0), b.edge_index.size(1)
    assert (N, E) == (51200, 153600)
    gi = build_index(b.edge_index.cuda(), N)
    torch.manual_seed(H)
    msg = torch.randn(E, H)
    ref = model_oracle.scatter(msg, b.edge_index[1], N, op)
    msg_csr = msg[gi.perm.cpu().long()].cuda()
    out = ops.segment_reduce(msg_csr, gi.rowptr, None, op)
    if op == "max":
        assert torch.equal(out.cpu(), ref)
    else:
        assert_close(out, ref, what=f"segsum cfg2 H={H}")


@pytest.mark.parametrize("op", ["max", "sum"])
def test_segreduce_stream_ragged_and_oversized_tiles(op):
    """N not a multiple of the 32-segment tile, empty segments, and tiles whose rows exceed the ring stage (a hub of
    in-degree 3000 and a run of degree-40 nodes): the global-memory fallback inside the streaming kernel."""
    g = torch.Generator().manual_seed(5)
    N = 4096 + 37
    degs = torch.randint(0, 6, (N,), generator=g)
    degs[100] = 3000
    degs[2000:2040] = 40
    degs[N - 1] = 0
    for H in (64, 128, 32):
        _seg_case(N, H, degs, op, seed=H)
    # every segment empty / every tile exactly full
    _seg_case(8192, 64, torch.zeros(8192, dtype=torch.int64), op)
    _seg_case(8192, 64, torch.full((8192,), 6, dtype=torch.int64), op)


# ------------------------------------------------------------------ tensor-core GEMMs at the benchmarked shapes
def _planes_case(M, K, H, seed):
    """x[M,K] . W4[4H,K]^T + b -> planes [4,M,H]; backward: dX out of the blocked planes, dW4 (TN) and db4."""
    from pert_gnn_kdd23_b200 import ops

    torch.manual_seed(seed)
    x = torch.randn(M, K)
    W = torch.randn(4 * H, K) / math.sqrt(K)
    b = torch.randn(4 * H)
    g = torch.randn(4, M, H)
    xd, Wd, bd = (t.double().requires_grad_() for t in (x, W, b))
    ref = torch.nn.functional.linear(xd, Wd, bd)
    rx, rW, rb = torch.autograd.grad(ref, (xd, Wd, bd), g.permute(1, 0, 2).reshape(M, 4 * H).double())
    xc, Wc, bc = (t.cuda().requires_grad_() for t in (x, W, b))
    planes = ops.linear(xc, Wc, bc, out_blocks=4)
    gx, gW, gb = torch.autograd.grad(planes, (xc, Wc, bc), g.cuda())
    tag = f"M={M} K={K} H={H}"
    # bars (norm-wise, against fp64): the tcgen05 kind::tf32 accumulator truncates (round toward zero) on every MMA, so
    # the error grows with the number of accumulation steps 3*K/8 (measured r2: 6e-7 at K=64, 2.5e-6 at K=256, 5e-6 at
    # K=512 -- DESIGN.md section 3); planes: K <= 144; dX: K = 4H; dW4: rows / CTA
    for got, want, what, tol in ((planes.permute(1, 0, 2).reshape(M, 4 * H), ref, "planes", 2e-6),
                                 (gx, rx, "dX", 4e-6 if H <= 64 else 8e-6), (gW, rW, "dW4", 3e-5), (gb, rb, "db4", 2e-5)):
        assert_close(got, want, rtol=tol, what=f"{what} {tag}", norm_only=True)
        assert_close(got, want, rtol=5 * tol, what=f"{what} {tag} (element-wise)")


@pytest.mark.parametrize("M", [4096, 51200, 102400])
@pytest.mark.parametrize("H", [64, 128])
def test_gemm_tensor_core_shapes(M, H):
    _planes_case(M, H, H, seed=M + H)


@pytest.mark.parametrize("H", [64, 128])
def test_gemm_tensor_core_conv0_width(H):
    """conv 0: K = round_up(9 + H, 8) (80 / 144), and a row count that is not a multiple of the 128-row tile."""
    _planes_case(51200 + 77, (9 + H + 7) // 8 * 8, H, seed=H)


@pytest.mark.parametrize("H", [64, 128])
def test_gemm_tn_fused_colsum(H):
    """pert_gemm_tn with a_colsum (what the engine calls: weight gradient + bias gradient in one pass)."""
    from pert_gnn_kdd23_b200 import _lib

    R, K = 51200, H
    torch.manual_seed(H)
    A = torch.randn(4, R, H).cuda()              # blocked [R, 4H]
    B = torch.randn(R, K).cuda()
    C = torch.zeros(4 * H, K).cuda()
    cs = torch.zeros(4 * H).cuda()
    _lib.call("pert_gemm_tn", A.data_ptr(), H, H, R * H, B.data_ptr(), K, 0, 0, C.data_ptr(), K, cs.data_ptr(), R,
              4 * H, K, torch.cuda.current_stream().cuda_stream)
    Ad = A.double().permute(1, 0, 2).reshape(R, 4 * H).cpu()
    assert_close(C, Ad.t() @ B.double().cpu(), rtol=2e-5, what=f"TN dW H={H}", norm_only=True)
    assert_close(cs, Ad.sum(0), rtol=2e-5, what=f"TN colsum H={H}", norm_only=True)


# ------------------------------------------------------------------ whole model at the real batch sizes
def _full_parity(cfg, ng, tag, grad_rtol=RTOL):
    """Outputs, loss, every gradient and the BatchNorm statistics of the FULL batch against the oracle.

    Derivatives are compared ON THE SAME LINEAR PIECE of the network.  A batch of 10^5 nodes puts ~10^7 arguments through
    the BatchNorm ReLUs; a few dozen of them lie within the 1e-6 by which two fp32 implementations of the conv stack differ,
    and each such unit that lands on the other side of zero adds or removes one node's term from weight-gradient sums whose
    result is ~sqrt(N) terms large -- 1e-3 of conv 0/1 gradients at cfg3-5 (measured: identical for the tcgen05, the exact
    fp32 SIMT GEMMs and both families of conv kernels, while BatchNorm itself agrees with torch to 1e-7:
    profiles/bn_probe.py), although every forward value agrees to 1e-6.  That is a property of fp32 evaluation of a
    piecewise-linear network, not of a kernel.  So the step ENGINE (what bench.py times) runs forward, the set of active ReLUs
    is read back from its saved activations (Engine.active_relus), and the oracle (fp32 = the reference path, fp64 =
    arbiter) is evaluated and differentiated with exactly those ReLUs active.  The free-running oracle (its own ReLUs) is
    checked on the forward values as well."""
    import copy

    from tests.helpers import assert_close_ref, assert_grads_close_ref

    b = make_batch(cfg, ng)
    a32 = forward_args(b)
    a64 = [t.double() if t.is_floating_point() else t for t in a32]
    oracle, model = make_models(cfg)
    oracle64 = copy.deepcopy(oracle).double()
    oracle_free = copy.deepcopy(oracle)
    oracle.train()
    oracle64.train()
    oracle_free.train()
    model.train()
    bc = b.to("cuda")

    def loss_of(g, l, y):
        return model_oracle.torch_quantile_loss(y, g.flatten(), 0.5) + 1e-3 * l.square().mean()

    gc, lc = model(*forward_args(bc))                      # engine path (model.use_engine is True)
    masks = {k: v.cpu() for k, v in model._engine.active_relus().items()}
    loss_c = loss_of(gc, lc, bc.y.float())
    loss_c.backward()
    go, lo = oracle(*a32, relu_masks=masks)
    go64, lo64 = oracle64(*a64, relu_masks=masks)
    loss_o, loss_64 = loss_of(go, lo, b.y.float()), loss_of(go64, lo64, b.y.double())
    loss_o.backward()
    loss_64.backward()
    assert_close_ref(gc, go, go64, what=f"{tag} global_predict")
    assert_close_ref(lc, lo, lo64, what=f"{tag} local_predict")
    assert_close_ref(loss_c, loss_o, loss_64, what=f"{tag} loss")
    assert_grads_close_ref(model.named_parameters(), oracle.named_parameters(), oracle64.named_parameters(), grad_rtol,
                           n_convs=len(model.convs))
    b64 = dict(oracle64.named_buffers())
    for n, bbuf in model.named_buffers():
        assert_close_ref(bbuf.float(), dict(oracle.named_buffers())[n].float(), b64[n].double(), what=f"{tag} {n}")
    # the free-running reference (its own ReLUs) gives the same forward values, and (almost) the same set of active ReLUs
    with torch.no_grad():
        gfree, lfree = oracle_free(*a32)
    assert_close(gc, gfree, what=f"{tag} global_predict (reference with its own ReLUs)")
    assert_close(lc, lfree, what=f"{tag} local_predict (reference with its own ReLUs)")
    # predicted-latency MAE of the batch (BASELINE north_star: "MAE matching the reference within 1e-4")
    mae_o = float((gfree.flatten() - b.y).abs().mean())
    mae_c = float((gc.detach().flatten() - bc.y).abs().mean())
    assert abs(mae_c - mae_o) <= 1e-4 * abs(mae_o), (mae_c, mae_o)


def test_model_cfg2_full():
    _full_parity(2, None, "cfg2[256]")


def test_model_cfg3_full():
    _full_parity(3, None, "cfg3[1024]")


def test_model_cfg4_shard():
    _full_parity(4, 512, "cfg4[512 of 4096]")


def test_model_cfg5_full():
    # 5 layers x 256,000 nodes x 128: outputs / loss / BN statistics at 1e-4; gradients at 2e-4 -- the truncating
    # tensor-core accumulators (DESIGN.md section 3) compound over ten GEMM layers of backward: measured <= 8.4e-5
    # (convs.3.lin_edge.weight; 1.9e-4 before the weight-gradient kernel rotated its chunks over several TMEM
    # accumulators) where the exact-fp32 reference path itself is 1.3e-5 from fp64 -- the bar leaves the run-to-run
    # spread of the float atomics (x1.5) above the measured value
    _full_parity(5, None, "cfg5[256x1000]", grad_rtol=2e-4)


def test_model_cfg2_jittered_sizes():
    """cfg2 with graph sizes 200 +- 20 % (no tile is a whole number of equal graphs): the graph-aligned tiles.
    Gradients are compared on the linear piece the engine's ReLUs selected, as in _full_parity: of the 2.4 M BatchNorm
    ReLUs of this batch, one argument lies within fp32 rounding of zero (1.1e-7, bn1, measured on a B200), the
    free-running oracle takes the other branch there, and that moves the gradients below that layer by ~1/sqrt(N)."""
    from pert_gnn_kdd23_b200.data import Batch
    from pert_gnn_kdd23_b200.synthetic import make_data_list

    oracle, model = make_models(2)
    b = Batch.from_data_list(make_data_list(2, num_graphs=96, jitter=0.2))
    oracle.train()
    model.train()
    go, lo = oracle(*forward_args(b))
    gc, lc = model(*forward_args(b.to("cuda")))
    assert_close(gc, go, what="cfg2j global_predict")
    masks = {k: v.cpu() for k, v in model._engine.active_relus().items()}
    go, lo = oracle(*forward_args(b), relu_masks=masks)
    loss_o = model_oracle.torch_quantile_loss(b.y.float(), go.flatten(), 0.5)
    loss_c = model_oracle.torch_quantile_loss(b.y.float().cuda(), gc.flatten(), 0.5)
    loss_o.backward()
    loss_c.backward()
    assert_grads_close(model.named_parameters(), oracle.named_parameters(), RTOL, n_convs=len(model.convs))


# ------------------------------------------------------------------ eval path (pert_gnn.py:254-294) on device accumulators
def test_eval_metrics_match_reference_loop():
    from pert_gnn_kdd23_b200.train import EvalMetrics, eval_step

    oracle, model = make_models(1)
    oracle.eval()
    model.eval()
    m = EvalMetrics("cuda", tau=0.95)
    mae = mape = q = 0.0
    n = 0
    for seed in range(3):
        b = make_batch(1, 48, seed=seed)
        with torch.no_grad():
            go, _ = oracle(*forward_args(b))
        p = go.flatten()
        mae += float((p - b.y).abs().sum())                 # pert_gnn.py:284-289
        mape += float(((p - b.y).abs() / b.y).sum())
        q += float(model_oracle.torch_quantile_loss(b.y.float(), p, 0.95) * b.y.shape[0])
        n += b.num_graphs
        assert eval_step(model, b.to("cuda"), 0.95, m) is None
    got = m.result()
    for a, r, what in zip(got, (mae / n, mape / n, q / n), ("mae", "mape", "qloss")):
        assert abs(a - r) <= 1e-4 * abs(r), (what, a, r)


# ------------------------------------------------------------------ A9: node_depth on the reference-generated goldens
def test_min_depth_and_node_depth_on_reference_goldens():
    """pert_min_depth + pert_node_depth + pert_level_order on the inputs of tests/golden/node_depth_*.npz (outputs of
    the reference's own misc.DFS / get_node_features / long cast, oracle/gen_golden.py), incl. the cycle and the
    unreachable-node cases; all nine graphs batched into ONE call as well as one by one."""
    import glob
    import os

    import numpy as np

    from oracle import index_oracle
    from pert_gnn_kdd23_b200.index import build_index, level_order, min_depth, node_depth

    files = sorted(glob.glob(os.path.join(os.path.dirname(__file__), "golden", "node_depth_*.npz")))
    assert len(files) == 9
    cases = [np.load(f) for f in files]
    eis, roots, ptr = [], [], [0]
    for c in cases:
        eis.append(torch.from_numpy(c["edge_index"]) + ptr[-1])
        roots.append(int(c["root"]) + ptr[-1])
        ptr.append(ptr[-1] + int(c["num_nodes"]))
    N = ptr[-1]
    gi = build_index(torch.cat(eis, 1).cuda(), N)
    gp = torch.tensor(ptr, dtype=torch.int32).cuda()
    d = min_depth(gp, gi, torch.tensor(roots, dtype=torch.int32).cuda())
    nd = node_depth(gp, d)
    lo = level_order(gp, d)
    assert nd.shape == (N, 1) and nd.dtype == torch.int64
    dn, ndn, lon = d.cpu().numpy(), nd.cpu().numpy(), lo.cpu().numpy()
    for i, c in enumerate(cases):
        sl = slice(ptr[i], ptr[i + 1])
        assert np.array_equal(dn[sl], c["min_depth"]), f"min_depth case {i}"
        assert np.array_equal(ndn[sl], c["node_depth"]), f"node_depth case {i}"
    assert np.array_equal(lon, index_oracle.level_order(np.array(ptr), dn))
    # single-graph calls (CTA-per-graph kernels with B = 1)
    for i, c in enumerate(cases):
        n = int(c["num_nodes"])
        g1 = build_index(torch.from_numpy(c["edge_index"]).cuda(), n)
        p1 = torch.tensor([0, n], dtype=torch.int32).cuda()
        d1 = min_depth(p1, g1, torch.tensor([int(c["root"])], dtype=torch.int32).cuda())
        assert np.array_equal(d1.cpu().numpy(), c["min_depth"])
        assert np.array_equal(node_depth(p1, d1).cpu().numpy(), c["node_depth"])


def test_node_depth_matches_generator_on_cfg3_batch():
    from pert_gnn_kdd23_b200.index import build_index, graph_ptr, min_depth, node_depth

    b = make_batch(3, 64)
    N, B = b.x.size(0), b.num_graphs
    gi = build_index(b.edge_index.cuda(), N)
    gp = graph_ptr(b.batch.cuda(), B)
    d = min_depth(gp, gi, b.ptr[:-1].to(torch.int32).cuda())
    assert torch.equal(node_depth(gp, d).cpu(), b.node_depth)


# ------------------------------------------------------------------ robustness (ADVICE.md round 1)
def test_train_step_with_fused_adam_really_updates_the_model():
    """train_step + FusedAdam(FlatParams(model)) (autograd path) == fused_train_step: the model must keep reading the
    flat buffer the optimizer updates (one FlatParams per model)."""
    import copy

    from pert_gnn_kdd23_b200.train import FlatParams, FusedAdam, fused_train_step, train_step

    _, model_a = make_models(1)
    model_b = copy.deepcopy(model_a)
    opt_a = FusedAdam(FlatParams(model_a), lr=1e-2)
    opt_b = FusedAdam(FlatParams(model_b), lr=1e-2)
    before = {n: p.detach().clone() for n, p in model_a.named_parameters()}
    for step in range(3):
        b = make_batch(1, 32, seed=step).to("cuda")
        la = train_step(model_a, opt_a, b, 0.5)
        lb = fused_train_step(model_b, opt_b, b, 0.5)
        assert_close(la.reshape(1), lb.reshape(1), what=f"loss step {step}")
    assert model_a._engine.fp is opt_a.fp
    moved = sum(float((p.detach() - before[n]).abs().max()) > 0 for n, p in model_a.named_parameters())
    assert moved >= len(before) - 4, f"only {moved} of {len(before)} parameters moved"
    pb = dict(model_b.named_parameters())
    for n, p in model_a.named_parameters():
        if n.endswith("lin_key.bias") or (n.endswith("lin_skip.bias") and not n.startswith("convs.1.")):
            continue
        assert_close(p, pb[n], rtol=2e-3, what=f"param {n}", norm_only=True)
    # optimizer created AFTER a first forward: the engine must adopt the new FlatParams, not keep its private one
    _, model_c = make_models(1)
    b = make_batch(1, 32, seed=0).to("cuda")
    model_c(*forward_args(b))
    opt_c = FusedAdam(FlatParams(model_c), lr=1e-2)
    w0 = model_c.global_linear1.weight.detach().clone()
    train_step(model_c, opt_c, b, 0.5)
    assert model_c._engine.fp is opt_c.fp
    assert float((model_c.global_linear1.weight.detach() - w0).abs().max()) > 0


def test_graph_replay_survives_workspace_growth():
    """Capture on a small batch, run a LARGER batch (the engine re-allocates its workspace), come back to the small
    one: the stale graph must not be replayed (ws_generation check) and the losses must match the eager path."""
    import copy

    from pert_gnn_kdd23_b200.train import FlatParams, FusedAdam, GraphedTrainStep, fused_train_step

    _, model_a = make_models(1)
    model_b = copy.deepcopy(model_a)
    opt_a = FusedAdam(FlatParams(model_a), lr=1e-3)
    opt_b = FusedAdam(FlatParams(model_b), lr=1e-3)
    small = make_batch(1, 16, seed=1).to("cuda")
    big = make_batch(1, 64, seed=2).to("cuda")
    gs = GraphedTrainStep(model_b, opt_b, 0.5)
    for it, data in enumerate([small, small, small, big, small, small, small, big, big, small]):
        la = fused_train_step(model_a, opt_a, data, 0.5)
        lb = gs(data)
        assert_close(lb, la, rtol=1e-4, what=f"loss step {it}", norm_only=True)
    assert gs.invalidations >= 1 and gs.capture_error is None
    assert gs.replays >= 2


def test_two_engines_on_two_streams_concurrently():
    """Two model replicas stepping at the same time on two streams of one device (tile-ticket ring, shared auxiliary
    stream): every replica must produce what it produces alone."""
    import copy

    from pert_gnn_kdd23_b200.train import FlatParams, FusedAdam, fused_train_step

    _, m0 = make_models(2)
    m1, r0, r1 = copy.deepcopy(m0), copy.deepcopy(m0), copy.deepcopy(m0)
    opts = [FusedAdam(FlatParams(m), lr=1e-3) for m in (m0, m1, r0, r1)]
    b0 = make_batch(2, 64, seed=1).to("cuda")
    b1 = make_batch(2, 64, seed=2).to("cuda")
    # reference: one after the other on the default stream
    ref0 = [float(fused_train_step(r0, opts[2], b0, 0.5)) for _ in range(4)]
    ref1 = [float(fused_train_step(r1, opts[3], b1, 0.5)) for _ in range(4)]
    torch.cuda.synchronize()
    s0, s1 = torch.cuda.Stream(), torch.cuda.Stream()
    l0, l1 = [], []
    for _ in range(4):
        with torch.cuda.stream(s0):
            l0.append(fused_train_step(m0, opts[0], b0, 0.5))
        with torch.cuda.stream(s1):
            l1.append(fused_train_step(m1, opts[1], b1, 0.5))
    torch.cuda.synchronize()
    for a, r in zip(l0, ref0):
        assert abs(float(a) - r) <= 1e-4 * abs(r), (float(a), r)
    for a, r in zip(l1, ref1):
        assert abs(float(a) - r) <= 1e-4 * abs(r), (float(a), r)


def test_runs_on_cuda1_while_cuda0_is_current():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    oracle, model = make_models(1)
    model = model.to("cuda:1")
    b = make_batch(1, 16)
    go, _ = oracle(*forward_args(b))
    assert torch.cuda.current_device() == 0
    gc, _ = model(*forward_args(b.to("cuda:1")))
    loss = gc.square().mean()
    loss.backward()
    assert gc.device.index == 1 and torch.cuda.current_device() == 0
    assert_close(gc, go, what="cuda:1 global_predict")
