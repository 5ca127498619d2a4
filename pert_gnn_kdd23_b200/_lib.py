"""ctypes binding of libpertgnn.so (the C-ABI declared in include/pertgnn.h).

There is NO fallback: if the shared library is missing or a call fails the
product path raises.  The library is built in-tree by ``__graft_entry__.build()``
(or ``make -C pert_gnn_kdd23_b200/csrc``).
"""
from __future__ import annotations

import ctypes as C
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libpertgnn.so")

P, I, LL, F, ULL = C.c_void_p, C.c_int, C.c_longlong, C.c_float, C.c_ulonglong

# name -> (restype, argtypes); must mirror include/pertgnn.h
SIGNATURES = {
    "pert_version": (I, []),
    "pert_index_workspace_bytes": (LL, [LL, LL]),
    "pert_build_index": (I, [P, P, I, LL, LL, I, I, P, P, P, P, P, P, P, P, P, LL, P, P]),
    "pert_graph_ptr": (I, [P, LL, LL, P, P, LL, P, P]),
    "pert_min_depth": (I, [P, LL, P, P, P, P, P]),
    "pert_node_depth": (I, [P, LL, P, P, P]),
    "pert_level_order": (I, [P, LL, P, P, P]),
    "pert_segment_reduce_fwd": (I, [P, P, P, P, LL, I, I, P]),
    "pert_segment_reduce_bwd": (I, [P, P, P, P, P, P, LL, I, I, P]),
    "pert_tconv_supported_width": (I, [I]),
    "pert_tconv_fwd": (I, [P, P, P, P, I, P, P, P, P, P, P, P, I, P, I, LL, LL, LL, I, P]),
    "pert_tconv_bwd": (I, [P, I, P, P, P, I, P, P, P, P, P, P, P, P, P, P, P, P, P, I, P, P, P, P, I, LL, LL, LL, I,
                           P]),
    "pert_gemm_nt": (I, [P, I, I, LL, P, I, P, P, I, I, LL, LL, I, I, I, I, P]),
    "pert_gemm_tn": (I, [P, I, I, LL, P, I, I, LL, P, I, P, LL, I, I, P]),
    "pert_colsum": (I, [P, I, I, LL, P, LL, I, P]),
    "pert_embedding_fwd": (I, [P, I, P, I, P, I, LL, I, I, P, P]),
    "pert_embedding_bwd": (I, [P, I, P, I, P, I, LL, I, P]),
    "pert_copy_cols": (I, [P, I, P, I, I, LL, P]),
    "pert_bn_workspace_bytes": (LL, [LL, I]),
    "pert_bn_fwd": (I, [P, I, P, P, P, P, P, F, F, I, I, P, P, P, I, LL, I, P, LL, P]),
    "pert_bn_bwd": (I, [P, I, P, I, P, I, P, P, P, I, I, P, I, P, P, P, LL, I, P]),
    "pert_pool_fwd": (I, [P, I, P, P, P, P, P, P, P, LL, LL, I, P, P]),
    "pert_pool_bwd": (I, [P, P, P, I, P, P, P, P, P, I, P, P, LL, LL, I, P]),
    "pert_relu_bwd": (I, [P, P, LL, P]),
    "pert_pinball_loss": (I, [P, P, F, LL, F, P, P, P]),
    "pert_eval_metrics": (I, [P, P, F, LL, P, P]),
    "pert_adam_step": (I, [P, P, P, P, LL, F, F, F, F, F, LL, F, P]),
    # fused all-reduce + Adam over peer memory (csrc/peer.cu)
    "pert_peer_exchange_bytes": (LL, [LL]),
    "pert_peer_alloc": (I, [LL, P, P]),
    "pert_peer_open": (I, [P, P]),
    "pert_peer_close": (I, [P]),
    "pert_peer_free": (I, [P]),
    "pert_allreduce_adam": (I, [P, P, P, P, LL, F, F, F, F, F, LL, F, P, I, I, P, P, P]),
    # device-side batch assembly from the pattern store (first / 7th argument: struct pointers, see store.py)
    "pert_store_assemble": (I, [P, P, LL, LL, LL, P, P, P, P]),
    # PERT-graph construction (pertgraph.py)
    "pert_pert_graph_count": (I, [P, LL, P, P, I, P, P, P]),
    "pert_pert_graph_build": (I, [P, LL, LL, P, P, P, P, P, P, P, P, I, I, P, P, P, P, P, P]),
    "pert_span_graph_count": (I, [P, LL, P, P, I, P, P, P]),
    "pert_span_graph_build": (I, [P, LL, LL, P, P, P, P, P, P, I, I, P, P, P, P, P, P]),
    # whole-model engine (first argument: const PertModelDesc*, see engine.py)
    "pert_model_workspace_bytes": (LL, [P, LL, LL, LL]),
    "pert_model_packed_bytes": (LL, [P]),
    "pert_model_workspace_offset": (LL, [P, LL, LL, LL, I, I]),
    "pert_model_forward": (I, [P, P, P, P, P, P, P, P, P, P, LL, LL, LL, P, P, P, P, P, LL, I, F, P, P, P, P, P, P,
                               P]),
    "pert_model_backward": (I, [P, P, P, P, P, P, P, P, LL, LL, LL, P, P, P, P, P, P, P, P, LL, I, F, P, P, P, P]),
    "pert_dropout_mask": (I, [LL, LL, I, LL, I, F, P, P]),
    # trace catalogue (catalogue.py)
    "pert_catalogue_run_flags": (I, [P, LL, P, P, P]),
    "pert_catalogue_summary": (I, [P, P, LL, P, P, P, P, P, P, ULL, ULL, P, P, P, P, P, P, P]),
    "pert_catalogue_verify": (I, [P, P, LL, P, P, P, P, P, P, P, P]),
    "pert_catalogue_rekey": (I, [P, P, LL, P, P, P, P, ULL, ULL, P, P]),
    "pert_catalogue_canon": (I, [P, P, LL, P, P, P]),
    "pert_catalogue_runtime_ids": (I, [P, P, LL, P, P]),
    "pert_catalogue_patterns": (I, [P, P, LL, P, LL, P, P, P, P]),
    "pert_catalogue_pairs": (I, [P, LL, LL, P, P, P, P, P, P, P, P, P]),
    "pert_catalogue_probs": (I, [P, P, LL, P, LL, LL, P, P, P]),
}

_lib = None


class PertGnnError(RuntimeError):
    pass


def lib():
    """Load (once) and return the ctypes handle; raises if the CUDA library is absent."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise PertGnnError(
                f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(there is no CPU / PyTorch fallback for the hot path)")
        h = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(h, name)
            fn.restype = res
            fn.argtypes = args
        _lib = h
    return _lib


def check(rc, what):
    if rc != 0:
        if rc > 0:
            raise PertGnnError(f"{what}: CUDA error {rc}")
        names = {-1: "bad argument", -2: "unsupported width/mode", -3: "index out of range",
                 -4: "a data-parallel peer never arrived (timeout)"}
        raise PertGnnError(f"{what}: {names.get(rc, rc)}")


def ptr(t):
    """Device pointer of a tensor (None -> NULL)."""
    if t is None:
        return None
    return t.data_ptr()


def stream():
    return torch.cuda.current_stream().cuda_stream


def on_device_of(fn):
    """Decorator: run ``fn`` with the CUDA device of its first CUDA-tensor argument current.  The C library launches
    on the current device and ``stream()`` returns that device's current stream, so every binding that takes tensors
    must pin the device (reference loop: ``--device N`` + ``model.to(f'cuda:{N}')`` never calls ``set_device``)."""
    import functools

    @functools.wraps(fn)
    def wrapped(*args, **kwargs):
        dev = None
        for a in args:
            if torch.is_tensor(a) and a.is_cuda:
                dev = a.device
                break
            d = getattr(a, "device", None)             # objects that carry a device (Engine, GraphIndex, FlatParams)
            if isinstance(d, torch.device) and d.type == "cuda":
                dev = d
                break
        if dev is None or dev.index is None or dev.index == torch.cuda.current_device():
            return fn(*args, **kwargs)
        with torch.cuda.device(dev):
            return fn(*args, **kwargs)

    return wrapped


def call(name, *args):
    rc = getattr(lib(), name)(*args)
    check(rc, name)
