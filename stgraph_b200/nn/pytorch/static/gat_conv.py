"""Vertex-centric GAT layer (mirror of ``stgraph/nn/pytorch/static/gat_conv.py:8-61``).

Same constructor, parameter / sub-module names (``fc``, ``attn_l``, ``attn_r``, ``feat_drop``,
``attn_drop``, ``leaky_relu``) and forward contract as the reference.

``softmax="stock"`` (default) traces the vertex program exactly as the reference ships it.
Because ``v.innbs`` is a one-element list, Python's ``max(embs)`` returns ``embs[0]`` and the trace
contains ``emb - emb``: the "edge softmax" is exactly a mean over in-neighbours, while the
backward still sends (reference-defined) gradients to ``attn_l`` / ``attn_r`` (SURVEY.md trap T2).
That behaviour is reproduced, not fixed.

``softmax="fused"`` is the genuine edge softmax (row-max subtraction, one-pass online softmax,
recompute-alpha backward, no ``[E,H]`` tensor and no atomics) on the hand-written kernels of
``csrc/gat.cu`` -- validated against a closed-form torch oracle, not against the reference.

Under ``torch.autocast`` the projection ``fc(feat)`` is bf16 / fp16.  The fused op and the stock program both read it as
it is and widen each element on load (fp32 softmax and output); the output is fp32 and the projection's gradient is
rounded to its dtype once.
"""
from __future__ import annotations

import torch
from torch import nn

from ....compiler import STGraph
from ....compiler.backend.pytorch.torch_callback import STGraphBackendTorch


_SOFTMAX_MODES = ("stock", "fused")


class GATConv(nn.Module):
    def __init__(self, in_feats, out_feats, num_heads, feat_drop=0.0, attn_drop=0.0, negative_slope=0.2,
                 activation=None, softmax: str = "stock"):
        super().__init__()
        if softmax not in _SOFTMAX_MODES:
            raise ValueError("softmax must be 'stock' or 'fused'")
        self.softmax = softmax
        self.activation = activation
        self.negative_slope = negative_slope
        self._in_feats, self._out_feats, self._num_heads = in_feats, out_feats, num_heads
        # parameter / sub-module names are the reference's, so its state_dicts load unchanged
        self.fc = nn.Linear(in_feats, num_heads * out_feats, bias=False)
        for name in ("attn_l", "attn_r"):
            self.register_parameter(name, nn.Parameter(torch.empty(num_heads, out_feats)))
        self.feat_drop, self.attn_drop = nn.Dropout(feat_drop), nn.Dropout(attn_drop)
        self.leaky_relu = nn.LeakyReLU(negative_slope)
        self.stgraph = STGraph(STGraphBackendTorch())
        self.reset_parameters()

    def reset_parameters(self):
        """Xavier-normal with the ReLU gain, in the reference's order (same values under the same seed)."""
        gain = nn.init.calculate_gain("relu")
        for weight in (self.fc.weight, self.attn_l, self.attn_r):
            nn.init.xavier_normal_(weight, gain=gain)

    def _scores(self, feat):
        """Per-head projections ``[N, H, D]`` and the two halves of the attention logit ``[N, H, 1]``."""
        proj = self.fc(self.feat_drop(feat)).view(-1, self._num_heads, self._out_feats)
        left = (proj * self.attn_l).sum(dim=-1, keepdim=True)
        right = (proj * self.attn_r).sum(dim=-1, keepdim=True)
        return proj, left, right

    def _stock_program(self):
        """The vertex program as the reference ships it (``gat_conv.py:48-56``), traced by our compiler.

        ``v.innbs`` is a one-element list while tracing, so ``max(logits)`` is ``logits[0]`` and the trace holds
        ``logit - logit`` (trap T2); the statement order below fixes the IR, which must equal the reference's."""
        # (the tracer patches this module's activation sub-modules while it runs: look `self.leaky_relu` up inside)

        @self.stgraph.compile(gnn_module=self)
        def nb_forward(v):
            logits = [nb.el + v.er for nb in v.innbs]
            top = max(logits)
            weights = [torch.exp(self.leaky_relu(x - top)) for x in logits]
            total = sum(weights)
            shares = [w / total for w in weights]
            rows = [nb.feat_src for nb in v.innbs]
            return sum([shares[k] * rows[k] for k in range(len(rows))])

        return nb_forward

    def forward(self, graph, feat):
        proj, left, right = self._scores(feat)
        if self.softmax == "fused":
            from ....ops_gat import gat_edge_softmax_aggregate

            out = gat_edge_softmax_aggregate(graph, left, right, proj, self.negative_slope)
        else:
            # Under autocast proj is bf16 / fp16 (el / er are fp32 by promotion): the VM reads it as it is, computes what
            # it computes on proj.float(), and the fp32 gradient it returns is rounded to proj's dtype by autograd.
            out = self._stock_program()(g=graph, n_feats={"el": left, "er": right, "feat_src": proj})
        return self.activation(out) if self.activation else out
