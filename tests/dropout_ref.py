"""Reference side of the dropout tests (test infrastructure, not a test module).

* ``philox4x32_10`` / ``keep_mask``: numpy restatement of the counter-based generator of the engine's fused dropout
  (include/pertgnn.h, pert_dropout_mask): Philox4x32-10 with key = (seed lo, seed hi) and counter = (j lo, j hi, layer,
  offset), j = the float4 index n * H/4 + c/4; word c % 4 drops unit (n, c) iff it is < floor(p * 2^32).
* ``DropoutOracle``: the CPU oracle of the model (oracle/model_oracle.py) with the dropout masks prescribed, so that
  it computes the same function as a dropout forward of the engine: ``F.dropout`` becomes ``x * keep / (1 - p)``.
"""
import math

import numpy as np
import torch
import torch.nn.functional as F

from oracle.model_oracle import OracleSAGEDeterministic, global_add_pool

M0, M1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
W0, W1 = 0x9E3779B9, 0xBB67AE85
_LO = np.uint64(0xFFFFFFFF)


def philox4x32_10(c0, c1, c2, c3, k0, k1):
    """Philox4x32-10 (Salmon et al., SC'11) over arrays: counter words c0..c3, key words k0, k1 (anything that
    broadcasts; values < 2^32).  Returns the four output words as uint32 arrays."""
    c = [np.asarray(v, dtype=np.uint64) for v in (c0, c1, c2, c3)]
    k0, k1 = int(k0), int(k1)
    for r in range(10):
        if r:
            k0, k1 = (k0 + W0) & 0xFFFFFFFF, (k1 + W1) & 0xFFFFFFFF
        p0 = M0 * c[0]            # exact: both factors < 2^32
        p1 = M1 * c[2]
        c = [(p1 >> np.uint64(32)) ^ c[1] ^ np.uint64(k0), p1 & _LO,
             (p0 >> np.uint64(32)) ^ c[3] ^ np.uint64(k1), p0 & _LO]
    return [v.astype(np.uint32) for v in c]


def threshold(p):
    """floor(p * 2^32) of the fp32 value of p, in double (what the library computes on the host)."""
    return math.floor(float(np.float32(p)) * 4294967296.0)


def keep_mask(seed, offset, layer, N, H, p):
    """bool [N, H]: True where unit (n, c) of BatchNorm ``layer`` is kept."""
    seed &= 0xFFFFFFFFFFFFFFFF
    offset &= 0xFFFFFFFFFFFFFFFF
    j = np.arange(N * (H // 4), dtype=np.uint64)
    words = philox4x32_10(j & _LO, j >> np.uint64(32), layer & 0xFFFFFFFF, offset & 0xFFFFFFFF,
                          seed & 0xFFFFFFFF, seed >> 32)
    t = threshold(p)
    keep = np.stack([w.astype(np.int64) >= t for w in words], axis=1)     # [N*H/4, 4]: column c = 4*(j % (H/4)) + k
    return keep.reshape(N, H)


class DropoutOracle(OracleSAGEDeterministic):
    """``forward(..., relu_masks=None, dropout_masks=None)``: with ``dropout_masks`` ({'bn{i}': [N,H] bool}) every
    ``F.dropout`` of the reference forward (model.py:103) is replaced by ``x * keep / (1 - p)``; with None it is the
    oracle's forward unchanged."""

    def forward(self, x, cat_X, edge_index, edge_attr, pattern_num_nodes, pattern_probs, entry_id, batch,
                relu_masks=None, dropout_masks=None):
        if dropout_masks is None:
            return super().forward(x, cat_X, edge_index, edge_attr, pattern_num_nodes, pattern_probs, entry_id, batch,
                                   relu_masks=relu_masks)
        relu = (lambda t, key: F.relu(t)) if relu_masks is None else (lambda t, key: t * relu_masks[key].to(t.dtype))
        cat_embeds = 0
        for i, emb in enumerate(self.cat_embedding):
            cat_embeds = cat_embeds + emb(cat_X[:, i])
        x = torch.cat([x, cat_embeds], dim=1)
        edge_embeds = torch.cat(
            [self.interface_embeds(edge_attr[:, 0]), self.rpctype_embeds(edge_attr[:, 1])], dim=1)
        for i, conv in enumerate(self.convs[:-1]):
            x = conv(x, edge_index, edge_embeds)
            x = self.bns[i](x)
            x = relu(x, f"bn{i}")
            if self.training and self.dropout > 0:
                x = x * dropout_masks[f"bn{i}"].to(x.dtype) / (1 - self.dropout)
        x = self.convs[-1](x, edge_index, edge_embeds)
        local_predict = self.local_linear(x)
        x = x * pattern_probs / pattern_num_nodes
        mean_x = global_add_pool(x, batch)
        g = torch.cat([mean_x, self.entry_embeds(entry_id)], dim=1)
        g = self.global_linear2(relu(self.global_linear1(g), "head"))
        return g, local_predict
