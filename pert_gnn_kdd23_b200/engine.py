"""Python side of the whole-model step engine (csrc/engine.cu): builds the ``PertModelDesc`` from a
``SAGEDeterministic`` module, owns the workspace, and exposes
  * ``Engine.forward`` / ``Engine.backward``  -- raw calls (no autograd), used by the fused train step;
  * ``engine_forward``                        -- a single autograd.Function for ``model.forward`` (drop-in path).
"""
from __future__ import annotations

import ctypes as C

import os

import torch

from . import _lib, ops
from .index import GraphIndex

MAX_CONVS, MAX_CAT = 8, 4
LL = C.c_longlong


class PertModelDesc(C.Structure):
    _fields_ = [
        ("F", C.c_int32), ("H", C.c_int32), ("n_convs", C.c_int32), ("n_cat", C.c_int32),
        ("cat_rows", C.c_int32 * MAX_CAT), ("n_entry", C.c_int32), ("n_if", C.c_int32), ("n_rpc", C.c_int32),
        ("k0", C.c_int32), ("bn_eps", C.c_float), ("bn_momentum", C.c_float),
        ("off_cat", LL * MAX_CAT), ("off_entry", LL), ("off_if", LL), ("off_rpc", LL),
        ("off_wq", LL * MAX_CONVS), ("off_bq", LL * MAX_CONVS), ("off_wk", LL * MAX_CONVS), ("off_bk", LL * MAX_CONVS),
        ("off_wv", LL * MAX_CONVS), ("off_bv", LL * MAX_CONVS), ("off_ws", LL * MAX_CONVS), ("off_bs", LL * MAX_CONVS),
        ("off_we", LL * MAX_CONVS), ("off_bn_g", LL * MAX_CONVS), ("off_bn_b", LL * MAX_CONVS),
        ("off_local_w", LL), ("off_local_b", LL), ("off_g1_w", LL), ("off_g1_b", LL), ("off_g2_w", LL),
        ("off_g2_b", LL),
    ]


def _bind():
    return _lib.lib()


class PertProbe(C.Structure):
    """Measurement probe (include/pertgnn.h): two CUDA events recorded around one kernel family of one layer."""
    _fields_ = [("kernel", C.c_int32), ("layer", C.c_int32), ("ev_start", C.c_void_p), ("ev_stop", C.c_void_p)]

    KERNELS = {"tconv_fwd": 1, "tconv_bwd": 2, "gemm_fwd": 3, "gemm_wgrad": 4, "gemm_dgrad": 5, "bn_apply": 6}
    _rt = None

    @classmethod
    def _cudart(cls):
        if cls._rt is None:
            import glob
            import os

            cands = glob.glob(os.path.join(os.path.dirname(torch.__file__), "lib", "libcudart*.so*")) + \
                glob.glob("/usr/local/cuda/lib64/libcudart.so*")
            if not cands:
                import nvidia.cuda_runtime as _n   # pip layout

                cands = glob.glob(os.path.join(os.path.dirname(_n.__file__), "lib", "libcudart.so*"))
            cls._rt = C.CDLL(sorted(cands)[0])
            cls._rt.cudaEventCreate.argtypes = [C.POINTER(C.c_void_p)]
            cls._rt.cudaEventElapsedTime.argtypes = [C.POINTER(C.c_float), C.c_void_p, C.c_void_p]
            cls._rt.cudaEventDestroy.argtypes = [C.c_void_p]
        return cls._rt

    @classmethod
    def create(cls, kernel, layer):
        rt = cls._cudart()
        a, b = C.c_void_p(), C.c_void_p()
        assert rt.cudaEventCreate(C.byref(a)) == 0 and rt.cudaEventCreate(C.byref(b)) == 0
        return cls(cls.KERNELS[kernel], layer, a, b)

    def elapsed_ms(self):
        ms = C.c_float()
        rc = self._cudart().cudaEventElapsedTime(C.byref(ms), self.ev_start, self.ev_stop)
        return ms.value if rc == 0 else float("nan")

    def destroy(self):
        rt = self._cudart()
        rt.cudaEventDestroy(self.ev_start)
        rt.cudaEventDestroy(self.ev_stop)


class Engine:
    """Owns flat parameters / gradients / BN buffers of one model replica and the engine workspace."""

    # launches per call (for the gpu_launches accounting of bench.py)
    def __init__(self, model, flat=None):
        from .train import FlatParams

        self.model = model
        self.fp = flat if flat is not None else FlatParams(model)
        self.lib = _bind()
        dev = self.fp.flat.device
        H = model.hidden_channels
        n_convs = len(model.convs)
        assert n_convs <= MAX_CONVS and len(model.cat_embedding) <= MAX_CAT
        # BN running statistics as one flat buffer; the module buffers become views of it
        n_bn = n_convs - 1
        self.bn_running = torch.empty(n_bn, 2, H, device=dev, dtype=torch.float32)
        self.bn_nbt = torch.zeros(n_bn, device=dev, dtype=torch.int64)
        for l, bn in enumerate(model.bns):
            self.bn_running[l, 0].copy_(bn.running_mean)
            self.bn_running[l, 1].copy_(bn.running_var)
            self.bn_nbt[l] = bn.num_batches_tracked
            bn._buffers["running_mean"] = self.bn_running[l, 0]
            bn._buffers["running_var"] = self.bn_running[l, 1]
            bn._buffers["num_batches_tracked"] = self.bn_nbt[l]
        d = PertModelDesc()
        d.F, d.H, d.n_convs, d.n_cat = model.in_channels, H, n_convs, len(model.cat_embedding)
        d.n_entry = model.entry_embeds.num_embeddings
        d.n_if = model.interface_embeds.num_embeddings
        d.n_rpc = model.rpctype_embeds.num_embeddings
        d.k0 = (model.in_channels + H + 7) // 8 * 8
        d.bn_eps = model.bns[0].eps
        d.bn_momentum = model.bns[0].momentum if model.bns[0].momentum is not None else 0.0
        base = self.fp.flat.data_ptr()

        def off(p):
            o = p.data_ptr() - base
            assert o % 16 == 0 and 0 <= o < self.fp.flat.numel() * 4, "parameter is not an aligned view of the flat buffer"
            return o // 4

        for i, e in enumerate(model.cat_embedding):
            d.cat_rows[i] = e.num_embeddings
            d.off_cat[i] = off(e.weight)
        d.off_entry, d.off_if, d.off_rpc = off(model.entry_embeds.weight), off(model.interface_embeds.weight), \
            off(model.rpctype_embeds.weight)
        for l, c in enumerate(model.convs):
            d.off_wq[l], d.off_bq[l] = off(c.lin_query.weight), off(c.lin_query.bias)
            d.off_wk[l], d.off_bk[l] = off(c.lin_key.weight), off(c.lin_key.bias)
            d.off_wv[l], d.off_bv[l] = off(c.lin_value.weight), off(c.lin_value.bias)
            d.off_ws[l], d.off_bs[l] = off(c.lin_skip.weight), off(c.lin_skip.bias)
            d.off_we[l] = off(c.lin_edge.weight)
        for l, bn in enumerate(model.bns):
            d.off_bn_g[l], d.off_bn_b[l] = off(bn.weight), off(bn.bias)
        d.off_local_w, d.off_local_b = off(model.local_linear.weight), off(model.local_linear.bias)
        d.off_g1_w, d.off_g1_b = off(model.global_linear1.weight), off(model.global_linear1.bias)
        d.off_g2_w, d.off_g2_b = off(model.global_linear2.weight), off(model.global_linear2.bias)
        self.desc = d
        self.n_convs = n_convs
        self.ws = None
        self.ws_key = (0, 0, 0)
        self.ws_generation = 0
        self._saved = None
        # dropout generator state (seed, offset), read by the BatchNorm kernels; every training forward with p > 0 adds 1
        # to the offset on the device (so a replayed CUDA graph draws fresh masks).  The seed is drawn from torch's
        # default generator at the first forward that needs it: a model without dropout never consumes random numbers.
        self.rng = torch.zeros(2, device=dev, dtype=torch.int64)
        self._rng_seeded = False

    # ------------------------------------------------------------------------------------------
    @property
    def device(self):
        return self.fp.flat.device

    def reserve(self, N, E, B):
        """Pre-size the workspace (growth only).  ``ws_generation`` changes whenever the buffer is re-allocated: a CUDA
        graph captured over the old buffer must not be replayed any more (train.GraphedTrainStep checks it)."""
        return self._workspace(int(N), int(E), int(B))

    def _workspace(self, N, E, B):
        if self.ws is None or N > self.ws_key[0] or E > self.ws_key[1] or B > self.ws_key[2]:
            key = (max(N, self.ws_key[0]), max(E, self.ws_key[1]), max(B, self.ws_key[2]))
            nbytes = self.lib.pert_model_workspace_bytes(C.byref(self.desc), *key)
            if nbytes < 0:
                _lib.check(int(nbytes), "pert_model_workspace_bytes")
            with torch.cuda.device(self.fp.flat.device):
                self.ws = torch.zeros(nbytes // 4, device=self.fp.flat.device, dtype=torch.float32)
            self.ws_key = key
            self.ws_generation += 1
        return self.ws

    def seed_dropout(self, seed, offset=0):
        """Sets the dropout generator state: the masks of a forward are a function of (seed, offset, layer) only."""
        seed = int(seed) & 0xFFFFFFFFFFFFFFFF
        if seed >= 1 << 63:
            seed -= 1 << 64                                  # the same 64 bits as an int64
        with torch.cuda.device(self.device):
            self.rng.copy_(torch.tensor([seed, int(offset)], dtype=torch.int64))
        self._rng_seeded = True

    @_lib.on_device_of
    def dropout_masks(self):
        """{'bn{i}': [N,H] bool}: the dropout keep masks of the LAST forward (all True when it applied no dropout), from
        pert_dropout_mask with the offset that forward used (read back from the device state).  Test aid, like
        ``active_relus``."""
        x, cat_X, entry_id, probs, pnn, batch, index, training, N, E, B, p = self._saved
        H = self.desc.H
        if not (training and p > 0):
            return {f"bn{l}": torch.ones(N, H, dtype=torch.bool, device=self.device) for l in range(self.n_convs - 1)}
        seed, offset = self.rng.tolist()
        out = {}
        for l in range(self.n_convs - 1):
            keep = torch.empty(N, H, dtype=torch.uint8, device=self.device)
            _lib.check(self.lib.pert_dropout_mask(seed, offset - 1, l, N, H, p, _lib.ptr(keep), _lib.stream()),
                       "pert_dropout_mask")
            out[f"bn{l}"] = keep.bool()
        return out

    def active_relus(self):
        """{'bn{i}': [N,H] bool, 'head': [B,H] bool}: which ReLUs were active in the LAST forward (read from the saved
        activations in the workspace; with dropout, a dropped unit reads as inactive).  Test aid: lets a reference be
        differentiated on the same linear piece."""
        x, cat_X, entry_id, probs, pnn, batch, index, training, N, E, B, p = self._saved
        H = self.desc.H
        out = {}
        for l in range(1, self.n_convs):
            off = self.lib.pert_model_workspace_offset(C.byref(self.desc), N, E, B, 0, l)
            _lib.check(int(min(off, 0)), "pert_model_workspace_offset")
            out[f"bn{l - 1}"] = self.ws[off:off + N * H].view(N, H) > 0
        off = self.lib.pert_model_workspace_offset(C.byref(self.desc), N, E, B, 1, 0)
        _lib.check(int(min(off, 0)), "pert_model_workspace_offset")
        out["head"] = self.ws[off:off + B * H].view(B, H) > 0
        return out

    def _pack_launches(self):
        # mirrors engine.cu: conv 0 contributes 24 segments, the others 16; a launch holds at most 96
        n, count = 0, 0
        for l in range(self.n_convs):
            count += 24 if l == 0 else 16
            if count + 24 > 96 or l == self.n_convs - 1:
                n, count = n + 1, 0
        return n

    def launches_forward(self):
        """Kernels pert_model_forward launches (memsets not counted): pack, edge tables (6 layers per launch),
        embeddings + copy, per conv GEMM + attention (whose epilogue also produces the BatchNorm statistics), per
        BatchNorm one apply kernel (dropout included), pool, head (which also advances the dropout offset)."""
        L = self.n_convs
        return self._pack_launches() + (L + 5) // 6 + self.desc.n_cat + 1 + 2 * L + (L - 1) + 1 + 1

    def launches_backward(self):
        """head, pool, per conv (target pass, source pass, weight GEMM, data GEMM), per BatchNorm reduce + apply,
        embedding scatters, edge-table gradients (3 layers per launch), unpack."""
        L = self.n_convs
        return 1 + 1 + 4 * L + 2 * (L - 1) + self.desc.n_cat + (L + 2) // 3 + self._pack_launches()

    @_lib.on_device_of
    def forward(self, x, cat_X, entry_id, probs, pnn, batch, index: GraphIndex, training, probe=None,
                index_ready=None):
        """-> (global_pred [B,1], local_pred [N,1]); keeps what backward needs in the workspace.  Training with
        ``model.dropout > 0`` applies dropout after every BatchNorm+ReLU (masks from ``self.rng``)."""
        N, E, B = x.size(0), index.E, entry_id.numel()
        p_drop = float(self.model.dropout)
        drop = bool(training) and p_drop > 0
        if drop and not self._rng_seeded:
            self.seed_dropout(int(torch.empty((), dtype=torch.int64).random_()))
        ws = self._workspace(N, E, B)
        dev = x.device
        x = x.contiguous().float()
        cat_X = cat_X.contiguous()
        entry_id = entry_id.contiguous().reshape(-1)
        probs = probs.reshape(-1).contiguous().float()
        pnn = pnn.reshape(-1).contiguous().float()
        batch = batch.contiguous()
        gpred = torch.empty(B, 1, device=dev, dtype=torch.float32)
        lpred = torch.empty(N, 1, device=dev, dtype=torch.float32)
        p = _lib.ptr
        rc = self.lib.pert_model_forward(
            C.byref(self.desc), p(self.fp.flat), p(self.bn_running), p(self.bn_nbt), p(x), p(cat_X), p(entry_id),
            p(probs), p(pnn), p(batch), N, E, B, p(index.rowptr), p(index.csr_src), p(index.csr_if), p(index.csr_rpc),
            p(ws), ws.numel() * 4, int(training), p_drop, p(self.rng) if drop else None, p(gpred), p(lpred),
            p(index.status),
            C.byref(probe) if probe is not None else None,
            C.c_void_p(index_ready.cuda_event) if index_ready is not None else None, _lib.stream())
        _lib.check(rc, "pert_model_forward")
        ops.LAUNCHES["n"] += self.launches_forward()
        self._saved = (x, cat_X, entry_id, probs, pnn, batch, index, bool(training), N, E, B, p_drop)
        return gpred, lpred

    @_lib.on_device_of
    def backward(self, d_global, d_local=None, grads=None, probe=None):
        """Accumulates (+=) parameter gradients into ``grads`` (default: the flat gradient buffer)."""
        x, cat_X, entry_id, probs, pnn, batch, index, training, N, E, B, p_drop = self._saved
        grads = self.fp.grad if grads is None else grads
        d_global = d_global.reshape(-1).contiguous().float()
        if d_local is not None:
            d_local = d_local.reshape(-1).contiguous().float()
        p = _lib.ptr
        ws = self.ws
        rc = self.lib.pert_model_backward(
            C.byref(self.desc), p(self.fp.flat), p(grads), p(cat_X), p(entry_id), p(probs), p(pnn), p(batch), N, E, B,
            p(index.rowptr), p(index.csr_src), p(index.csr_if), p(index.csr_rpc), p(index.colptr), p(index.csc_pos),
            p(index.csc_dst), p(ws), ws.numel() * 4, int(training), p_drop, p(d_global), p(d_local),
            C.byref(probe) if probe is not None else None, _lib.stream())
        _lib.check(rc, "pert_model_backward")
        ops.LAUNCHES["n"] += self.launches_backward()


# PERT_DIRECT_GRADS=0: always hand the parameter gradients to autograd (A/B of the host-side cost, see _EngineFn.backward)
_DIRECT_GRADS = os.environ.get("PERT_DIRECT_GRADS", "1") != "0"


class _EngineFn(torch.autograd.Function):
    """model.forward as ONE autograd node: inputs are the parameters (so autograd routes their gradients),
    outputs (global_pred, local_pred)."""

    @staticmethod
    def forward(ctx, engine, x, cat_X, entry_id, probs, pnn, batch, index, training, *params):
        g, l = engine.forward(x, cat_X, entry_id, probs, pnn, batch, index, training)
        ctx.engine = engine
        ctx.token = engine._saved
        return g, l

    @staticmethod
    def backward(ctx, dg, dl):
        eng = ctx.engine
        if eng._saved is not ctx.token:
            raise RuntimeError("engine workspace was overwritten by a later forward before this backward ran "
                               "(one in-flight forward per model replica)")
        gbuf = torch.zeros_like(eng.fp.flat)
        eng.backward(dg, dl, grads=gbuf)
        eng.last_grad_buffer = gbuf      # every parameter gradient is a view of this buffer (one all-reduce in DP)
        views = eng.fp.views_of(gbuf)
        params = eng.fp.params
        if _DIRECT_GRADS:
            # The reference loop calls optimizer.zero_grad() (set_to_none) before every backward (pert_gnn.py:232): every
            # .grad is None and autograd's AccumulateGrad would just install the 42 views one by one (~0.25 ms of host
            # time per step, a third of this loop's budget).  In exactly that state -- no gradient to accumulate into,
            # no hooks registered on any parameter -- the views are attached directly and autograd gets no parameter
            # gradients to route.  Any other state takes the regular autograd path below.
            direct = True
            for p in params:
                if p.grad is not None or p._backward_hooks or getattr(p, "_post_accumulate_grad_hooks", None):
                    direct = False
                    break
            if direct:
                for p, v in zip(params, views):
                    p.grad = v
                return (None,) * (9 + len(params))
        return (None,) * 9 + tuple(views)


def engine_forward(engine, x, cat_X, entry_id, probs, pnn, batch, index, training):
    return _EngineFn.apply(engine, x, cat_X, entry_id, probs, pnn, batch, index, training, *engine.fp.params)
