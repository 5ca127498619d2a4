"""``SAGEDeterministic`` -- drop-in for reference model.py:10-114.

Same constructor arguments, same ``forward(x, cat_X, edge_index, edge_attr, pattern_num_nodes,
pattern_probs, entry_id, batch) -> (global_predict [B,1], local_predict [N,1])``, same parameter /
buffer names (``state_dict`` keys) and same layer-count quirk (``max(2, num_layers)`` convs,
SURVEY.md fact 4), so ``pert_gnn.py``'s train loop (``model(...)``, ``loss.backward()``,
``torch.optim.Adam(model.parameters())``) runs unchanged.  All compute is libpertgnn CUDA kernels.
"""
from __future__ import annotations

import torch
import torch.nn.functional as F

from . import ops
from .index import cached_index
from .nn import BatchNorm1d, Linear, TransformerConv


class SAGEDeterministic(torch.nn.Module):
    def __init__(self, in_channels, cat_dims, entry_id_max, interface_id_max, rpctype_id_max,
                 hidden_channels, num_layers, dropout):
        super().__init__()
        H = hidden_channels
        self.in_channels, self.hidden_channels = in_channels, H
        self.convs = torch.nn.ModuleList()
        self.convs.append(TransformerConv(in_channels + H, H, heads=1, edge_dim=2 * H))
        self.bns = torch.nn.ModuleList()
        self.bns.append(BatchNorm1d(H))
        for _ in range(num_layers - 2):
            self.convs.append(TransformerConv(H, H, heads=1, edge_dim=2 * H))
            self.bns.append(BatchNorm1d(H))
        self.convs.append(TransformerConv(H, H, heads=1, edge_dim=2 * H))
        self.local_linear = Linear(H, 1)
        self.global_linear1 = Linear(2 * H, H)
        self.global_linear2 = Linear(H, 1)
        self.cat_embedding = torch.nn.ModuleList([torch.nn.Embedding(n, H) for n in cat_dims])
        self.dropout = dropout
        self.entry_embeds = torch.nn.Embedding(entry_id_max + 1, H)
        self.interface_embeds = torch.nn.Embedding(interface_id_max + 1, H)
        self.rpctype_embeds = torch.nn.Embedding(rpctype_id_max + 1, H)
        self.edge_linear = Linear(-1, 2 * H)   # lazy + unused in the reference forward (model.py:68): bias only
        # True: whole forward/backward issued by the C++ step engine (csrc/engine.cu); False: one autograd
        # Function per operator (ops.py).  Same kernels, same results; the engine removes the interpreter gaps.  (Dropout:
        # the engine draws its own counter-based masks, the operator path calls F.dropout -- same distribution.)
        self.use_engine = True
        self._engine = None
        # test hook (operator path only): dict that receives the post-ReLU activations ('bn{i}', 'head'), so that a reference
        # can be differentiated on the SAME linear piece of the network (tests/test_gpu_fullsize.py); None = off
        self._capture = None

    def engine(self, flat=None):
        """The step engine of this replica.  There is ONE FlatParams per model: the one passed in, else the one a
        ``FlatParams(model)`` (e.g. an optimizer's) registered on the module, else a new one -- never a second flat
        buffer behind the back of an optimizer.  Re-created only if the parameters moved (``.to()``, ``load``)."""
        from .engine import Engine
        from .train import FlatParams

        eng = self._engine
        if flat is None:
            if eng is not None and eng.fp.owns_fast():      # per-step path: two pointer checks instead of one per parameter
                return eng
            reg = self.__dict__.get("_flat_params")
            flat = reg if (reg is not None and reg.owns(self)) else FlatParams(self, bind_grads=False)
        if eng is not None and eng.fp is flat and flat.owns(self):
            return eng
        if not flat.owns(self):
            raise RuntimeError("the FlatParams handed to model.engine() no longer holds this model's parameters "
                               "(the model was moved or re-flattened after the optimizer was built)")
        self._engine = Engine(self, flat)
        return self._engine

    def reset_parameters(self):
        for conv in self.convs:
            conv.reset_parameters()
        for bn in self.bns:
            bn.reset_parameters()

    def forward(self, x, cat_X, edge_index, edge_attr, pattern_num_nodes, pattern_probs, entry_id, batch,
                index=None):
        H, Fin = self.hidden_channels, self.in_channels
        N = x.size(0)
        if index is None:
            index = cached_index(edge_index, N, edge_attr, self.interface_embeds.num_embeddings,
                                 self.rpctype_embeds.num_embeddings)
        index.num_graphs = entry_id.numel()
        if self.use_engine:
            # training dropout (model.py:103) runs inside the engine's BatchNorm kernels (Engine.forward)
            from .engine import engine_forward

            return engine_forward(self.engine(), x, cat_X, entry_id, pattern_probs, pattern_num_nodes, batch, index,
                                  self.training)
        # prologue (model.py:87-90): internal layout [cat_embeds | x | pad]; conv 0 weights permuted to match
        h = ops.embed_concat(x, cat_X, [e.weight for e in self.cat_embedding])
        pad = h.size(1) - (Fin + H)
        perm0 = torch.cat([torch.arange(Fin, Fin + H), torch.arange(0, Fin)]).to(x.device)
        if_t, rpc_t = self.interface_embeds.weight, self.rpctype_embeds.weight
        for i, conv in enumerate(self.convs[:-1]):
            h = conv.forward_tables(h, index, if_t, rpc_t, perm0 if i == 0 else None, pad if i == 0 else 0)
            h = self.bns[i](h, relu=True)
            if self._capture is not None:
                self._capture[f"bn{i}"] = h.detach()
            h = F.dropout(h, p=self.dropout, training=self.training)
        last = len(self.convs) - 1
        h = self.convs[-1].forward_tables(h, index, if_t, rpc_t, perm0 if last == 0 else None,
                                          pad if last == 0 else 0)
        B = entry_id.numel()
        pool, local_predict = ops.pool_local(h, pattern_probs, pattern_num_nodes, batch,
                                             self.local_linear.weight, self.local_linear.bias, B)
        g = torch.cat([pool, ops.embedding(self.entry_embeds.weight, entry_id.reshape(-1))], dim=1)
        g = ops.linear(g, self.global_linear1.weight, self.global_linear1.bias, relu=True)
        if self._capture is not None:
            self._capture["head"] = g.detach()
        g = ops.linear(g, self.global_linear2.weight, self.global_linear2.bias)
        return g, local_predict
