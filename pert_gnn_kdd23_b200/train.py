"""Train / eval step mirroring reference pert_gnn.py:191-193 (pinball loss), :213-251 (train), :254-294 (test),
plus the data-parallel wrapper the reference lacks (SURVEY.md 8e: shard independent graphs over GPUs, ONE
flat-buffer gradient all-reduce per step).
"""
from __future__ import annotations

import torch
import torch.distributed as dist

from . import _lib, ops


def torch_quantile_loss(y_test, y_hat, tau):
    """reference pert_gnn.py:191-193."""
    e = y_test - y_hat
    return torch.mean(torch.maximum(tau * e, (tau - 1) * e))


def model_inputs(data):
    """Argument tuple of SAGEDeterministic.forward from a Batch (pert_gnn.py:233-243); the per-node pattern
    probability ``rt_probs`` is precomputed at collation instead of rebuilt on the host every step (:220-230)."""
    probs = data.rt_probs if "rt_probs" in data else data.pattern_probs
    return (data.x, data.cat_X, data.edge_index, data.edge_attr, data.pattern_num_nodes, probs, data.entry_id,
            data.batch)


class FlatParams:
    """All parameters (and their gradients) of a module as views into two flat fp32 buffers, so that the
    gradient all-reduce and the Adam update are ONE collective and ONE kernel (payload <= 4.8 MB, latency-bound)."""

    def __init__(self, module, bind_grads=True):
        params = [p for p in module.parameters() if p.requires_grad]
        al = lambda k: (k + 63) // 64 * 64          # every parameter starts on a 256-byte boundary (float4 / TMA)
        n = sum(al(p.numel()) for p in params)
        dev = params[0].device
        self.flat = torch.zeros(n, device=dev, dtype=torch.float32)
        self.grad = torch.zeros(n, device=dev, dtype=torch.float32)
        off = 0
        self._layout = []                              # (offset, shape, contiguous strides) of every parameter
        for p in params:
            k = p.numel()
            self.flat[off:off + k].copy_(p.data.reshape(-1))
            p.data = self.flat[off:off + k].view_as(p)
            if bind_grads:
                p.grad = self.grad[off:off + k].view_as(p)
            self._layout.append((off, tuple(p.shape), tuple(p.stride())))
            off += al(k)
        self.params = params
        self.numel = n
        # ONE FlatParams per module: model.engine() adopts this one instead of re-pointing p.data into a second flat
        # buffer (which would silently detach an optimizer built over this one)
        if isinstance(module, torch.nn.Module):
            module.__dict__["_flat_params"] = self

    @property
    def device(self):
        return self.flat.device

    def owns(self, module):
        """True while every trainable parameter of ``module`` is still a view into this flat buffer."""
        lo = self.flat.data_ptr()
        hi = lo + self.flat.numel() * 4
        ps = [p for p in module.parameters() if p.requires_grad]
        return len(ps) == len(self.params) and all(lo <= p.data_ptr() < hi for p in ps)

    def owns_fast(self):
        """Cheap form of ``owns`` for the per-step path: the first and the last parameter still live in the flat buffer
        (``module.to()`` / re-flattening moves all of them; ``load_state_dict`` copies in place)."""
        lo = self.flat.data_ptr()
        hi = lo + self.flat.numel() * 4
        return lo <= self.params[0].data_ptr() < hi and lo <= self.params[-1].data_ptr() < hi

    def views_of(self, buf):
        """One view per parameter (its shape) into ``buf``, a flat tensor laid out like ``flat`` / ``grad``."""
        return [buf.as_strided(shape, stride, off) for off, shape, stride in self._layout]

    def zero_grad(self):
        self.grad.zero_()


class FusedAdam:
    """torch.optim.Adam(params, lr) semantics (reference pert_gnn.py:343) in one kernel over FlatParams."""

    def __init__(self, flat: FlatParams, lr=3e-4, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.0):
        self.fp = flat
        self.lr, self.betas, self.eps, self.wd = lr, betas, eps, weight_decay
        self.m = torch.zeros_like(flat.flat)
        self.v = torch.zeros_like(flat.flat)
        self.t = 0

    @property
    def device(self):
        return self.fp.flat.device

    def zero_grad(self, set_to_none=False):
        self.fp.zero_grad()

    @_lib.on_device_of
    def step(self, grad_scale=1.0):
        self.t += 1
        _lib.call("pert_adam_step", _lib.ptr(self.fp.flat), _lib.ptr(self.fp.grad), _lib.ptr(self.m),
                  _lib.ptr(self.v), self.fp.numel, self.lr, self.betas[0], self.betas[1], self.eps, self.wd, self.t,
                  float(grad_scale), _lib.stream())
        ops.LAUNCHES["n"] += 1


class PeerAdam(FusedAdam):
    """FusedAdam whose step also averages the gradient over the data-parallel ranks: ONE kernel per step
    (csrc/peer.cu) that publishes the flat gradient in a CUDA-IPC exchange buffer, reduces + updates ITS 1/world slice
    of the parameters from the peers' buffers over NVLink and pushes the result to every rank (m, v are maintained
    for the owned slice only) -- no NCCL call on the step path.  ``DataParallel`` skips its own
    all-reduce when the optimiser is a PeerAdam.  Needs one process per GPU on one node (``torch.distributed``
    initialised, used once to exchange the 64-byte IPC handles); with a single rank it degenerates to FusedAdam."""

    fused_allreduce = True

    def __init__(self, flat: FlatParams, lr=3e-4, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.0, group=None):
        super().__init__(flat, lr, betas, eps, weight_decay)
        import ctypes

        self.group = group
        self.world = dist.get_world_size(group) if dist.is_initialized() else 1
        self.rank = dist.get_rank(group) if dist.is_initialized() else 0
        self._own = None
        self._peers = []
        self.status = torch.zeros(1, dtype=torch.int32, device=flat.flat.device)
        self.timing = torch.zeros(5, dtype=torch.int64, device=flat.flat.device)   # ns publish/wait/reduce/gather, calls
        if self.world == 1:
            return
        if self.world > 8:
            raise _lib.PertGnnError("PeerAdam supports up to 8 ranks on one node")
        L = _lib.lib()
        dev = flat.flat.device

        def all_ok(ok):
            # every rank takes part in every collective of the setup, whatever happened locally: a rank that failed
            # must not leave the others waiting in a different collective
            t = torch.tensor([1.0 if ok else 0.0], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MIN, group=group)
            return float(t) > 0.0

        err = None
        handle = (ctypes.c_ubyte * 64)()
        try:
            nbytes = L.pert_peer_exchange_bytes(flat.numel)
            own = ctypes.c_void_p()
            _lib.check(L.pert_peer_alloc(nbytes, ctypes.byref(own), handle), "pert_peer_alloc")
            self._own = own.value
        except Exception as e:  # noqa: BLE001
            err = e
        if not all_ok(err is None):
            self.close(collective=False)
            raise _lib.PertGnnError(f"PeerAdam setup failed on some rank (local error: {err!r})")
        mine = torch.tensor(list(handle), dtype=torch.uint8, device=dev)
        gathered = [torch.empty_like(mine) for _ in range(self.world)]
        dist.all_gather(gathered, mine, group=group)
        ptrs = []
        try:
            for r in range(self.world):
                if r == self.rank:
                    ptrs.append(self._own)
                    continue
                hb = (ctypes.c_ubyte * 64)(*gathered[r].cpu().tolist())
                pp = ctypes.c_void_p()
                _lib.check(L.pert_peer_open(hb, ctypes.byref(pp)), "pert_peer_open")
                self._peers.append(pp.value)
                ptrs.append(pp.value)
        except Exception as e:  # noqa: BLE001
            err = e
        if not all_ok(err is None):
            self.close(collective=False)
            raise _lib.PertGnnError(f"PeerAdam peer mapping failed on some rank (local error: {err!r})")
        self._xbufs = (ctypes.c_void_p * self.world)(*ptrs)
        dist.barrier(group=group)      # every rank has mapped every buffer before the first step touches them

    @_lib.on_device_of
    def step(self, grad_scale=1.0):
        if self.world == 1:
            return super().step(grad_scale)
        self.t += 1
        _lib.call("pert_allreduce_adam", _lib.ptr(self.fp.flat), _lib.ptr(self.fp.grad), _lib.ptr(self.m),
                  _lib.ptr(self.v), self.fp.numel, self.lr, self.betas[0], self.betas[1], self.eps, self.wd, self.t,
                  float(grad_scale), self._xbufs, self.rank, self.world, _lib.ptr(self.status), _lib.ptr(self.timing),
                  _lib.stream())
        ops.LAUNCHES["n"] += 1

    def phase_times_us(self, reset=True):
        """Mean microseconds CTA 0 of the fused kernel spent publishing, waiting for the peers' gradients, reducing +
        Adam on its slice + pushing the parameters, and gathering the peers' slices (synchronising read; the wait phase
        is the slowest rank's skew plus the flag round trip over NVLink)."""
        t = self.timing.cpu().tolist()
        if reset:
            self.timing.zero_()
        n = max(t[4], 1)
        return {"publish_us": t[0] / n / 1e3, "wait_us": t[1] / n / 1e3, "reduce_adam_us": t[2] / n / 1e3,
                "gather_us": t[3] / n / 1e3, "calls": t[4]}

    def check(self):
        """Synchronising check of the device status word (a peer that never arrived sets PERT_ERR_PEER_TIMEOUT)."""
        code = int(self.status.item())
        if code != 0:
            _lib.check(code, "pert_allreduce_adam")

    def close(self, collective=True):
        L = _lib.lib()
        for pp in self._peers:
            L.pert_peer_close(pp)
        self._peers = []
        if self._own:
            if collective and dist.is_initialized() and self.world > 1:
                torch.cuda.synchronize()
                dist.barrier(group=self.group)     # nobody still reads this buffer
            L.pert_peer_free(self._own)
            self._own = None


class DataParallel:
    """One process per GPU; each rank owns a shard of the graphs; gradients are averaged with a single
    all-reduce of the flat gradient buffer (NCCL over NVLink on the box, gloo in the CPU tests).
    BatchNorm statistics stay per-replica (like DDP); parity claims are per shard (DESIGN.md)."""

    def __init__(self, flat: FlatParams, group=None):
        self.fp = flat
        self.group = group
        self.world = dist.get_world_size(group) if dist.is_initialized() else 1

    def all_reduce_grads(self, optimizer=None):
        """Sums the flat gradient over the ranks (unless ``optimizer`` does it itself, see PeerAdam) and returns the
        scale that turns the sum into the mean."""
        if self.world > 1 and not getattr(optimizer, "fused_allreduce", False):
            dist.all_reduce(self.fp.grad, op=dist.ReduceOp.SUM, group=self.group)
        return 1.0 / self.world


    def all_reduce_module_grads(self, model):
        """Averages the gradients ATTACHED to the parameters (``p.grad``) over the ranks -- the torch-optimizer branch
        of ``train_step``: ``torch.optim``'s ``zero_grad()`` defaults to ``set_to_none=True``, so the views FlatParams
        bound to ``fp.grad`` are gone and autograd installs views of the engine's last gradient buffer instead.  One
        all-reduce of that buffer when every gradient is a view of it, else flatten -> reduce -> scatter back."""
        if self.world <= 1:
            return
        gs = [p.grad for p in model.parameters() if p.grad is not None]
        if not gs:
            return
        gb = getattr(getattr(model, "_engine", None), "last_grad_buffer", None)
        if gb is not None:
            lo, hi = gb.data_ptr(), gb.data_ptr() + gb.numel() * gb.element_size()
            if all(lo <= g.data_ptr() < hi for g in gs):
                dist.all_reduce(gb, op=dist.ReduceOp.SUM, group=self.group)
                gb.mul_(1.0 / self.world)
                return
        flat = torch.cat([g.reshape(-1) for g in gs])
        dist.all_reduce(flat, op=dist.ReduceOp.SUM, group=self.group)
        flat.mul_(1.0 / self.world)
        o = 0
        for g in gs:
            g.copy_(flat[o:o + g.numel()].view_as(g))
            o += g.numel()


def train_step(model, optimizer, data, tau=0.5, dp: DataParallel | None = None):
    """One iteration of the loop body of reference pert_gnn.py:231-247 on a device-resident Batch.
    Returns the (device) loss tensor; no host sync."""
    fused = isinstance(optimizer, FusedAdam)
    if fused and hasattr(model, "engine"):
        # the model must read the SAME flat buffer the optimizer updates, and its p.grad must be the views of fp.grad
        eng = model.engine(optimizer.fp)
        lo, hi = optimizer.fp.grad.data_ptr(), optimizer.fp.grad.data_ptr() + optimizer.fp.grad.numel() * 4
        for p in optimizer.fp.params:
            if p.grad is None or not (lo <= p.grad.data_ptr() < hi):
                base = optimizer.fp.flat.data_ptr()
                o = (p.data_ptr() - base) // 4
                p.grad = optimizer.fp.grad[o:o + p.numel()].view_as(p)
    optimizer.zero_grad()
    global_pred, _ = model(*model_inputs(data))
    loss = torch_quantile_loss(data.y.float(), global_pred.flatten(), tau)
    loss.backward()
    if fused:
        scale = dp.all_reduce_grads(optimizer) if dp is not None else 1.0
        optimizer.step(grad_scale=scale)
    else:
        if dp is not None:
            dp.all_reduce_module_grads(model)
        optimizer.step()
    return loss


_SIDE_STREAMS = {}


def _side_stream(device):
    key = torch.device(device).index
    st = _SIDE_STREAMS.get(key)
    if st is None:
        st = _SIDE_STREAMS[key] = torch.cuda.Stream(device)
    return st


@_lib.on_device_of
def _fused_fwd_bwd(model, optimizer: FusedAdam, data, tau, index, probe, use_index_cache=True):
    """Device work of one step up to the gradients: (index build) -> zero grads -> engine forward -> pinball loss +
    its gradient -> engine backward into the flat gradient buffer.  Returns (loss [1], index)."""
    from .index import build_index, cached_index

    eng = model.engine(optimizer.fp) if (model._engine is None or model._engine.fp is not optimizer.fp) \
        else model._engine
    x, cat_X, edge_index, edge_attr, pnn, probs, entry_id, batch = model_inputs(data)
    index_ready = None
    if index is None:
        n_if, n_rpc = model.interface_embeds.num_embeddings, model.rpctype_embeds.num_embeddings
        if use_index_cache:
            index = cached_index(edge_index, x.size(0), edge_attr, n_if, n_rpc)
        else:
            # build the index on a side stream: the forward only waits for it right before the first attention
            # kernel, so it overlaps the parameter pack, the input prologue and the first GEMM
            main = torch.cuda.current_stream(x.device)
            side = _side_stream(x.device)
            side.wait_stream(main)
            with torch.cuda.stream(side):
                index = build_index(edge_index, x.size(0), edge_attr, n_if, n_rpc, check=False)
                index_ready = torch.cuda.Event()
                index_ready.record(side)
    optimizer.zero_grad()
    with torch.no_grad():
        gpred, _ = eng.forward(x, cat_X, entry_id, probs, pnn, batch, index, model.training, probe=probe,
                               index_ready=index_ready)
        B = gpred.size(0)
        loss = torch.empty(1, device=gpred.device, dtype=torch.float32)
        dy = torch.empty(B, device=gpred.device, dtype=torch.float32)
        _lib.call("pert_pinball_loss", _lib.ptr(data.y), _lib.ptr(gpred), float(tau), B, 1.0, _lib.ptr(loss),
                  _lib.ptr(dy), _lib.stream())
        ops.LAUNCHES["n"] += 1
        eng.backward(dy, None, probe=probe)
    return loss, index


def fused_train_step(model, optimizer: FusedAdam, data, tau=0.5, dp: DataParallel | None = None, index=None,
                     probe=None):
    """Same step as ``train_step`` but without autograd: engine forward -> pinball loss + its gradient (one
    kernel) -> engine backward into the flat gradient buffer -> (all-reduce) -> fused Adam.  5 C calls per step.
    Returns the device loss tensor [1]."""
    loss, _ = _fused_fwd_bwd(model, optimizer, data, tau, index, probe)
    with torch.no_grad():
        scale = dp.all_reduce_grads(optimizer) if dp is not None else 1.0
        optimizer.step(grad_scale=scale)
    return loss


class GraphedTrainStep:
    """``fused_train_step`` with the device work up to the gradients replayed from a CUDA graph.

    One graph per (input buffers, shapes) key -- e.g. one per slab of ``data.DevicePrefetcher``'s ring, or one per
    resident batch.  The graph holds: index build, gradient zeroing, engine forward, pinball loss, engine backward
    (~45 kernel launches become one ``cudaGraphLaunch``: no per-kernel launch gaps on the GPU, ~0.5 ms less host
    work per step).  The gradient all-reduce and Adam (its step count is a by-value kernel argument) are issued
    eagerly after the replay.  The first step on a new key runs eagerly (it also does the library's one-time
    initialisation), the second is captured; a key whose capture fails stays eager.  The reference has no
    counterpart (its loop body, pert_gnn.py:231-247, launches every operator from Python each step)."""

    def __init__(self, model, optimizer: FusedAdam, tau=0.5, dp: DataParallel | None = None, max_graphs=32):
        self.model, self.opt, self.tau, self.dp = model, optimizer, tau, dp
        self.max_graphs = max_graphs
        self._seen = {}      # key -> "ran-once" | "failed" | entry dict
        self.capture_error = None
        self.replays = 0
        self.invalidations = 0

    @staticmethod
    def _key(data):
        # every tensor the captured kernels read must sit where it sat at capture time
        ptrs = tuple(t.data_ptr() for t in model_inputs(data) if torch.is_tensor(t)) + (data.y.data_ptr(),)
        return ptrs + (tuple(data.x.shape), int(data.edge_index.size(1)), int(data.num_graphs))

    def _finish(self, loss):
        with torch.no_grad():
            scale = self.dp.all_reduce_grads(self.opt) if self.dp is not None else 1.0
            self.opt.step(grad_scale=scale)
        return loss

    def __call__(self, data):
        # the dropout threshold and scale are by-value kernel arguments: frozen in a captured graph
        key = self._key(data) + (float(self.model.dropout),)
        ent = self._seen.get(key, "unseen")
        if isinstance(ent, dict):
            pass
        elif ent == "ran-once" and len(self._seen) <= self.max_graphs:
            ent = self._capture(data, key)
        else:
            if ent == "unseen":
                self._seen[key] = "ran-once"
            ent = None
        if isinstance(ent, dict) and ent["ws_gen"] != ent["engine"].ws_generation:
            # the engine re-allocated its workspace since the capture (a bigger batch came by): the captured kernels
            # point into freed memory -> drop EVERY graph of that generation and start over on the eager path
            self._seen = {k: "ran-once" for k in self._seen}
            self.invalidations += 1
            ent = None
        if not isinstance(ent, dict):          # eager: first visit, capture failed, or too many keys
            loss, _ = _fused_fwd_bwd(self.model, self.opt, data, self.tau, None, None)
            return self._finish(loss)
        ent["graph"].replay()
        ops.LAUNCHES["n"] += ent["launches"]
        self.replays += 1
        return self._finish(ent["loss"])

    def _capture(self, data, key):
        g = torch.cuda.CUDAGraph()
        l0 = ops.LAUNCHES["n"]
        try:
            with torch.cuda.graph(g):
                # the index is rebuilt inside the graph: the same buffers may hold another batch at replay time
                loss, index = _fused_fwd_bwd(self.model, self.opt, data, self.tau, None, None, use_index_cache=False)
        except Exception as e:  # noqa: BLE001 - any capture failure leaves this key on the eager path
            self.capture_error = repr(e)
            ops.LAUNCHES["n"] = l0
            self._seen[key] = "failed"
            torch.cuda.synchronize()
            return None
        n = ops.LAUNCHES["n"] - l0
        ops.LAUNCHES["n"] = l0
        eng = self.model._engine
        ent = {"graph": g, "loss": loss, "index": index, "data": data, "launches": n, "engine": eng,
               "ws_gen": eng.ws_generation, "ws": eng.ws}       # "ws" keeps the captured workspace alive
        self._seen[key] = ent
        return ent


class AsyncLossReader:
    """Per-step loss read-back that does not drain the stream: ``push(loss)`` enqueues a 4-byte D2H copy into a pinned
    slot + an event right behind the step that produced ``loss`` and returns the value of the PREVIOUS push (whose
    copy has long finished while the current step was being enqueued); ``flush()`` returns the last one.  The
    reference reads ``loss.item()`` synchronously every step (pert_gnn.py:248); the running sum is identical, the GPU
    just never waits for the host between steps."""

    def __init__(self, device):
        self.buf = torch.zeros(2, dtype=torch.float32).pin_memory()
        self.ev = [torch.cuda.Event(), torch.cuda.Event()]
        self.pending = None
        self.n = 0
        self.device = device

    def push(self, loss):
        slot = self.n & 1
        self.n += 1
        self.buf[slot:slot + 1].copy_(loss.detach().reshape(1), non_blocking=True)
        self.ev[slot].record()
        prev = self.flush() if self.pending is not None else None
        self.pending = slot
        return prev

    def flush(self):
        if self.pending is None:
            return None
        self.ev[self.pending].synchronize()
        v = float(self.buf[self.pending])
        self.pending = None
        return v


class EvalMetrics:
    """Device-side accumulators of the reference's eval loop (pert_gnn.py:254-294): sum |pred - y|, sum |pred - y| / y
    and sum of the per-graph pinball terms, kept in three doubles ON THE DEVICE (``pert_eval_metrics``) so that a
    whole epoch needs ONE D2H read (``result()``) instead of the reference's per-batch syncs."""

    def __init__(self, device, tau=0.5):
        self.acc = torch.zeros(3, dtype=torch.float64, device=device)
        self.tau = float(tau)
        self.count = 0

    @property
    def device(self):
        return self.acc.device

    def reset(self):
        self.acc.zero_()
        self.count = 0

    @_lib.on_device_of
    def update(self, y, yhat):
        y = y.contiguous()
        yhat = yhat.reshape(-1).contiguous().float()
        _lib.call("pert_eval_metrics", _lib.ptr(y), _lib.ptr(yhat), self.tau, y.numel(), _lib.ptr(self.acc),
                  _lib.stream())
        ops.LAUNCHES["n"] += 1
        self.count += int(y.numel())

    def result(self):
        """-> (mae, mape, quantile loss), each divided by the number of graphs seen, like pert_gnn.py:290-294."""
        a = self.acc.cpu()
        n = max(self.count, 1)
        return float(a[0]) / n, float(a[1]) / n, float(a[2]) / n


@torch.no_grad()
def eval_step(model, data, tau=0.5, metrics: EvalMetrics | None = None):
    """Loop body of reference pert_gnn.py:260-289 on a device-resident Batch: engine forward (eval mode: BatchNorm
    running statistics), then the three sums on the device.  With ``metrics`` the sums are accumulated there and
    nothing is returned to the host; without, returns the device tensor [3] (mae, mape, quantile loss * B)."""
    global_pred, _ = model(*model_inputs(data))
    m = metrics if metrics is not None else EvalMetrics(global_pred.device, tau)
    m.update(data.y, global_pred)
    return m.acc if metrics is None else None


@torch.no_grad()
def evaluate(model, loader, device, tau=0.5):
    """reference ``test(loader)`` (pert_gnn.py:254-294): model.eval(), every batch through eval_step, one read-back."""
    was_training = model.training
    model.eval()
    m = EvalMetrics(device, tau)
    for data in loader:
        eval_step(model, data.to(device), tau, m)
    model.train(was_training)
    return m.result()
