"""Training-mode dropout of the step engine (model.py:103, fused into the BatchNorm-apply kernel).

CPU: the numpy Philox4x32-10 against the Random123 known-answer vectors, the threshold edge cases and drop rates, host-
side argument checks of the C-ABI, the dropout-aware oracle.  GPU (-m gpu): pert_dropout_mask bit for bit against the
numpy restatement, the saved activations of a dropout forward, full cfg2 / cfg3 parity with the oracle evaluated on the
engine's masks, drop-in vs fused step, graph replay (device-side offset advance), eval mode and seeding."""
import copy
import ctypes as C
import math

import numpy as np
import pytest
import torch

from tests.dropout_ref import DropoutOracle, keep_mask, philox4x32_10, threshold
from tests.helpers import RTOL, assert_grads_close, elem_err, forward_args, make_batch

P_DROP = 0.1


def _within_6_sigma(k, n, p):
    return abs(k / n - p) <= 6.0 * math.sqrt(p * (1.0 - p) / n)


# ================================================================== CPU
@pytest.mark.parametrize("counter,key,want", [
    ((0, 0, 0, 0), (0, 0), (0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8)),
    ((0xFFFFFFFF,) * 4, (0xFFFFFFFF,) * 2, (0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD)),
    ((0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344), (0xA4093822, 0x299F31D0),
     (0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1)),
])
def test_philox_known_answers(counter, key, want):
    got = tuple(int(w[()]) for w in philox4x32_10(*counter, *key))
    assert got == want, [hex(v) for v in got]


def test_threshold_edges_and_drop_rate():
    N, H = 51200, 64                               # 3.3 M units (one cfg2 BatchNorm output)
    assert keep_mask(9, 0, 0, N, H, 0.0).all()
    assert not keep_mask(9, 0, 0, N, H, 1.0).any()
    assert threshold(0.0) == 0 and threshold(1.0) == 2 ** 32
    for p in (0.1, 0.5):
        keep = keep_mask(12345, 3, 1, N, H, p)
        assert _within_6_sigma(int((~keep).sum()), keep.size, p), (p, 1 - keep.mean())
    # the layer and the offset are counter words: different masks
    a, b, c = keep_mask(1, 0, 0, 64, 64, 0.5), keep_mask(1, 0, 1, 64, 64, 0.5), keep_mask(1, 1, 0, 64, 64, 0.5)
    assert not np.array_equal(a, b) and not np.array_equal(a, c)


def _cpu_desc():
    from pert_gnn_kdd23_b200.engine import Engine
    from pert_gnn_kdd23_b200.model import SAGEDeterministic
    from pert_gnn_kdd23_b200.synthetic import model_args

    return Engine(SAGEDeterministic(*model_args(1))).desc


@pytest.mark.parametrize("p", [-0.1, 1.5, float("nan")])
def test_abi_rejects_bad_dropout_before_any_launch(p):
    """Non-NULL stand-in pointers everywhere: the only bad argument is p, and the call must refuse before any launch."""
    from pert_gnn_kdd23_b200 import _lib

    L = _lib.lib()
    assert L.pert_version() >= 2004
    d = C.byref(_cpu_desc())
    fake = 4096
    fwd = lambda p_, rng: L.pert_model_forward(d, *([fake] * 9), 100, 200, 4, *([fake] * 5), 1 << 40, 1, p_, rng,
                                              fake, fake, fake, None, None, None)
    bwd = lambda p_: L.pert_model_backward(d, *([fake] * 7), 100, 200, 4, *([fake] * 8), 1 << 40, 1, p_, fake, None,
                                          None, None)
    assert fwd(p, fake) == -1
    assert bwd(p) == -1
    assert L.pert_dropout_mask(1, 0, 0, 8, 64, p, fake, None) == -1
    # training with p > 0 needs the generator state
    assert fwd(0.5, None) == -1


def test_dropout_mask_rejects_bad_shapes():
    from pert_gnn_kdd23_b200 import _lib

    L = _lib.lib()
    assert L.pert_dropout_mask(1, 0, 0, -1, 64, 0.1, 4096, None) == -1
    assert L.pert_dropout_mask(1, 0, 0, 8, 66, 0.1, 4096, None) == -1
    assert L.pert_dropout_mask(1, 0, 0, 8, 64, 0.1, None, None) == -1
    assert L.pert_dropout_mask(1, 0, 0, 0, 64, 0.1, 4096, None) == 0        # nothing to do: no launch


def _oracle_pair(p, seed=0):
    from oracle.model_oracle import OracleSAGEDeterministic
    from pert_gnn_kdd23_b200.synthetic import model_args

    args = model_args(1)[:-1] + (p,)
    torch.manual_seed(seed)
    base = OracleSAGEDeterministic(*args)
    new = DropoutOracle(*args)
    new.load_state_dict(base.state_dict())
    return base, new


def test_oracle_dropout_masks(monkeypatch):
    from oracle import model_oracle

    b = make_batch(1, 8)
    p = 0.3
    base, new = _oracle_pair(p)
    base.train()
    new.train()
    # None: the oracle unchanged (same torch dropout draws)
    torch.manual_seed(5)
    g0, l0 = base(*forward_args(b))
    torch.manual_seed(5)
    g1, l1 = new(*forward_args(b))
    assert torch.equal(g0, g1) and torch.equal(l0, l1)
    # all-True masks: dropout degenerates to the 1/(1-p) scaling
    N, H = b.x.size(0), new.bns[0].num_features
    ones = {f"bn{i}": torch.ones(N, H, dtype=torch.bool) for i in range(len(new.bns))}
    g2, l2 = new(*forward_args(b), dropout_masks=ones)
    monkeypatch.setattr(model_oracle.F, "dropout", lambda x, p, training: x / (1 - p) if training else x)
    g3, l3 = base(*forward_args(b))
    assert torch.allclose(g2, g3, rtol=1e-6, atol=1e-6) and torch.allclose(l2, l3, rtol=1e-6, atol=1e-6)


# ================================================================== GPU
def _model(cfg, p, seed=0):
    from pert_gnn_kdd23_b200.model import SAGEDeterministic
    from pert_gnn_kdd23_b200.synthetic import model_args

    torch.manual_seed(seed)
    return SAGEDeterministic(*(model_args(cfg)[:-1] + (p,))).cuda()


def _saved_acts(eng):
    """The post-BatchNorm(-ReLU-dropout) activations x[1..L-1] of the engine's last forward (copies)."""
    x, cat_X, entry_id, probs, pnn, batch, index, training, N, E, B, p = eng._saved
    H = eng.desc.H
    out = []
    for l in range(1, eng.n_convs):
        off = eng.lib.pert_model_workspace_offset(C.byref(eng.desc), N, E, B, 0, l)
        assert off >= 0
        out.append(eng.ws[off:off + N * H].view(N, H).clone())
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("N,H", [(51200, 64), (256000, 128), (1, 64), (7, 64), (51201, 64)])
def test_mask_kernel_matches_numpy(N, H):
    from pert_gnn_kdd23_b200 import _lib

    keep = torch.empty(N, H, dtype=torch.uint8, device="cuda")
    for seed, offset, layer, p in ((0, 0, 0, 0.1), (-1, 7, 1, 0.5), (0x123456789ABCDEF, (1 << 32) + 3, 2, 0.1),
                                   (2024, 11, 4, 0.3)):
        _lib.call("pert_dropout_mask", seed, offset, layer, N, H, p, keep.data_ptr(), _lib.stream())
        want = keep_mask(seed, offset, layer, N, H, p)
        assert np.array_equal(keep.cpu().numpy().astype(bool), want), (seed, offset, layer, p)


@pytest.mark.gpu
def test_engine_forward_applies_the_mask():
    """cfg2, p = 0.1: dropped units of every saved activation are exactly 0; the kept units of the first BatchNorm
    output equal scale x their p = 0 value; the drop rate among active ReLUs is p."""
    bc = make_batch(2).to("cuda")
    model = _model(2, 0.0)
    model.train()
    eng = model.engine()
    with torch.no_grad():
        model(*forward_args(bc))
    y0 = _saved_acts(eng)
    model.dropout = P_DROP
    eng.seed_dropout(1234, 5)
    with torch.no_grad():
        model(*forward_args(bc))
    y1 = _saved_acts(eng)
    masks = eng.dropout_masks()
    assert eng.rng.tolist() == [1234, 6]
    scale = float(np.float32(1.0 / (1.0 - np.float32(P_DROP))))
    for l, y in enumerate(y1):
        keep = masks[f"bn{l}"]
        assert not bool(y[~keep].any()), f"bn{l}: a dropped unit is not 0"
    keep0 = masks["bn0"]
    assert elem_err(y1[0][keep0], y0[0][keep0] * scale) <= 1e-6
    active = y0[0] > 0
    n_act = int(active.sum())
    dropped = int((active & ~keep0).sum())
    assert _within_6_sigma(dropped, n_act, P_DROP), (dropped, n_act)


def _dropout_parity(cfg, tag):
    """_full_parity of tests/test_gpu_fullsize.py with p = 0.1: the oracle (fp32 reference path and fp64 arbiter) is
    evaluated on the engine's ReLU pattern AND its dropout masks."""
    from oracle import model_oracle
    from pert_gnn_kdd23_b200.model import SAGEDeterministic
    from pert_gnn_kdd23_b200.synthetic import model_args
    from tests.helpers import assert_close_ref, assert_grads_close_ref

    b = make_batch(cfg)
    a32 = forward_args(b)
    a64 = [t.double() if t.is_floating_point() else t for t in a32]
    args = model_args(cfg)[:-1] + (P_DROP,)
    torch.manual_seed(0)
    oracle = DropoutOracle(*args)
    model = SAGEDeterministic(*args)
    model.load_state_dict(oracle.state_dict())
    model = model.cuda()
    oracle64 = copy.deepcopy(oracle).double()
    for m in (oracle, oracle64, model):
        m.train()
    bc = b.to("cuda")

    def loss_of(g, l, y):
        return model_oracle.torch_quantile_loss(y, g.flatten(), 0.5) + 1e-3 * l.square().mean()

    model.engine().seed_dropout(99 + cfg, 0)
    gc, lc = model(*forward_args(bc))
    relu = {k: v.cpu() for k, v in model._engine.active_relus().items()}
    drop = {k: v.cpu() for k, v in model._engine.dropout_masks().items()}
    assert all(0 < float((~v).float().mean()) < 2 * P_DROP for v in drop.values())
    loss_c = loss_of(gc, lc, bc.y.float())
    loss_c.backward()
    go, lo = oracle(*a32, relu_masks=relu, dropout_masks=drop)
    go64, lo64 = oracle64(*a64, relu_masks=relu, dropout_masks=drop)
    loss_o, loss_64 = loss_of(go, lo, b.y.float()), loss_of(go64, lo64, b.y.double())
    loss_o.backward()
    loss_64.backward()
    assert_close_ref(gc, go, go64, what=f"{tag} global_predict")
    assert_close_ref(lc, lo, lo64, what=f"{tag} local_predict")
    assert_close_ref(loss_c, loss_o, loss_64, what=f"{tag} loss")
    assert_grads_close_ref(model.named_parameters(), oracle.named_parameters(), oracle64.named_parameters(), RTOL,
                           n_convs=len(model.convs))
    b32, b64 = dict(oracle.named_buffers()), dict(oracle64.named_buffers())
    for n, bbuf in model.named_buffers():
        assert_close_ref(bbuf.float(), b32[n].float(), b64[n].double(), what=f"{tag} {n}")


@pytest.mark.gpu
def test_dropout_parity_cfg2_full():
    _dropout_parity(2, "cfg2[256] p=0.1")


@pytest.mark.gpu
def test_dropout_parity_cfg3_full():
    _dropout_parity(3, "cfg3[1024] p=0.1")


def _twins(cfg, p):
    a = _model(cfg, p)
    b = _model(cfg, p, seed=1)
    b.load_state_dict(a.state_dict())
    a.train()
    b.train()
    return a, b


@pytest.mark.gpu
def test_dropin_and_fused_step_agree():
    """Same seed and offset: model(...) + loss.backward() and fused_train_step draw the same masks and give the same
    gradient; both run the engine (the drop-in forward records its call in the engine).  The two runs differ only in the
    order of float atomics, which moved small entries of convs.1.lin_value.weight by 1.4e-5 (elem_err) and the
    cancellation-limited convs.1.lin_key.weight by 1.3e-6 of its largest entry (B200), so the gradients are held to the
    project's parity bars (tests/helpers.py:assert_grads_close); a different mask would move them by O(1)."""
    from pert_gnn_kdd23_b200.train import FlatParams, FusedAdam, fused_train_step, torch_quantile_loss

    bc = make_batch(2).to("cuda")
    ma, mb = _twins(2, P_DROP)
    ea = ma.engine()
    ea.seed_dropout(7, 3)
    ea._saved = None
    gp, _ = ma(*forward_args(bc))
    assert ea._saved is not None and ea._saved[-1] == P_DROP, "the drop-in forward did not run the engine"
    torch_quantile_loss(bc.y.float(), gp.flatten(), 0.5).backward()
    fp = FlatParams(mb)
    opt = FusedAdam(fp, lr=3e-4)
    eb = mb.engine(fp)
    eb.seed_dropout(7, 3)
    eb._saved = None
    fused_train_step(mb, opt, bc)
    assert eb._saved is not None
    assert ea.rng.tolist() == eb.rng.tolist() == [7, 4]
    ka, kb = ea.dropout_masks(), eb.dropout_masks()
    assert all(torch.equal(ka[k], kb[k]) for k in ka)
    assert_grads_close(ma.named_parameters(), mb.named_parameters(), RTOL, n_convs=len(ma.convs))


@pytest.mark.gpu
def test_graph_replay_draws_fresh_masks():
    """GraphedTrainStep (the offset advances on the device inside the replayed graph) against fused_train_step (eager)
    for 6 steps from the same seed: same offsets, same masks, same losses; consecutive masks are independent."""
    from pert_gnn_kdd23_b200.train import FlatParams, FusedAdam, GraphedTrainStep, fused_train_step

    bc = make_batch(2).to("cuda")
    ma, mb = _twins(2, P_DROP)
    fa, fb = FlatParams(ma), FlatParams(mb)
    oa, ob = FusedAdam(fa, lr=3e-4), FusedAdam(fb, lr=3e-4)
    ea, eb = ma.engine(fa), mb.engine(fb)
    ea.seed_dropout(31, 0)
    eb.seed_dropout(31, 0)
    gstep = GraphedTrainStep(ma, oa)
    prev = None
    for s in range(6):
        la = float(gstep(bc))
        lb = float(fused_train_step(mb, ob, bc))
        assert ea.rng.tolist() == eb.rng.tolist() == [31, s + 1]
        ka, kb = ea.dropout_masks(), eb.dropout_masks()
        for k in ka:
            assert torch.equal(ka[k], kb[k]), f"step {s} {k}"
        assert abs(la - lb) <= 1e-5 * abs(lb), (s, la, lb)
        if prev is not None:
            for k in ka:
                both = int((~ka[k] & ~prev[k]).sum())
                assert not torch.equal(ka[k], prev[k])
                assert _within_6_sigma(both, ka[k].numel(), P_DROP * P_DROP), (s, k, both)
        prev = ka
    assert gstep.replays == 5 and gstep.capture_error is None


@pytest.mark.gpu
def test_eval_mode_and_seeding():
    """eval: p = 0.5 is the p = 0 forward bit for bit and leaves the offset alone; the same seed gives the same masks;
    p = 0 never draws from torch's generator (a model without dropout keeps the user's random stream)."""
    bc = make_batch(2, 64).to("cuda")
    model = _model(2, 0.5)
    eng = model.engine()
    eng.seed_dropout(5, 2)
    model.eval()
    with torch.no_grad():
        g5, l5 = model(*forward_args(bc))
        y5 = _saved_acts(eng)
        model.dropout = 0.0
        g0, l0 = model(*forward_args(bc))
        y0 = _saved_acts(eng)
    assert eng.rng.tolist() == [5, 2]
    assert all(torch.equal(a, b) for a, b in zip(y5, y0))
    assert elem_err(g5, g0) <= 1e-6 and elem_err(l5, l0) <= 1e-6
    # same seed and offset -> same masks
    model.train()
    model.dropout = 0.5
    runs = []
    for _ in range(2):
        eng.seed_dropout(77, 0)
        with torch.no_grad():
            model(*forward_args(bc))
        runs.append(eng.dropout_masks())
    assert all(torch.equal(runs[0][k], runs[1][k]) for k in runs[0])
    # lazy seed: drawn from torch's default generator at the first forward that needs it, never before
    fresh = _model(2, 0.0)
    fresh.train()
    torch.manual_seed(3)
    with torch.no_grad():
        fresh(*forward_args(bc))
    r1 = torch.rand(4)
    torch.manual_seed(3)
    assert torch.equal(r1, torch.rand(4)) and not fresh._engine._rng_seeded
    fresh.dropout = 0.2
    torch.manual_seed(3)
    with torch.no_grad():
        fresh(*forward_args(bc))
    assert fresh._engine._rng_seeded and fresh._engine.rng.tolist()[1] == 1


@pytest.mark.gpu
def test_p_one_drops_everything():
    bc = make_batch(2, 32).to("cuda")
    model = _model(2, 1.0)
    model.train()
    gp, _ = model(*forward_args(bc))
    gp.sum().backward()
    assert all(not bool(y.any()) for y in _saved_acts(model._engine))
    assert all(not bool(v.any()) for v in model._engine.dropout_masks().values())
    assert all(bool(torch.isfinite(p.grad).all()) for p in model.parameters() if p.grad is not None)
