"""Temporal GCN cell (mirror of ``stgraph/nn/pytorch/temporal/tgcn.py:5-55``).

Three ``GCNConv`` + three ``Linear(2H, H)`` GRU gates; module names (``conv_z/r/h``,
``linear_z/r/h``) match the reference so state_dicts interchange.  The graph convolutions are
clamped to +-1e6 exactly like the reference.

``fused=True`` keeps the parameters and the math but runs the three graph convolutions as ONE
GEMM ``X @ [W_z | W_r | W_h]`` and ONE aggregation of width 3H (every output column of a GEMM / of
the aggregation is computed independently, so the values are the same as three separate
convolutions up to cuBLAS tiling), the gates as GEMMs on column blocks (no concatenations) and the
element-wise work as three fused passes (bias + clamp, reset gate, update gate + candidate state)
instead of ~16 torch kernels, with no tracing or executor work per step; a whole BPTT window can
be captured in a CUDA graph (SURVEY.md section 8(f).1).  The whole cell is one autograd op with a
hand-written backward (``ops_tgcn``); ``fused="pieces"`` chains the same kernels through torch
autograd piece by piece (``ops_gcn`` / ``ops_gru``), which costs about three times the launches.
"""
import torch

from ..static.gcn_conv import GCNConv


class TGCN(torch.nn.Module):
    def __init__(self, in_channels, out_channels, fused: bool | str | None = None):
        """``fused=None`` (default): run the fused cell whenever it computes the same thing as the three separate
        convolutions (always, for the cell as the reference builds it: the convolutions share the graph, ``X`` and
        ``norm``); ``fused=False`` forces the reference-structured path (three traced vertex programs through the
        executor: 1216 ms instead of ~200 ms per WikiMaths epoch), ``fused=True`` forces the fused one."""
        super().__init__()
        self.in_channels = in_channels
        self.out_channels = out_channels
        self.fused = fused
        self.conv_z = GCNConv(self.in_channels, self.out_channels, activation=None)
        self.linear_z = torch.nn.Linear(2 * self.out_channels, self.out_channels)
        self.conv_r = GCNConv(self.in_channels, self.out_channels, activation=None)
        self.linear_r = torch.nn.Linear(2 * self.out_channels, self.out_channels)
        self.conv_h = GCNConv(self.in_channels, self.out_channels, activation=None)
        self.linear_h = torch.nn.Linear(2 * self.out_channels, self.out_channels)

    def __getstate__(self):
        # the parameter pack of the fused cell holds non-leaf tensors: never part of a copy / pickle of the module
        state = self.__dict__.copy()
        state.pop("_pack_cache", None)
        return state

    def _set_hidden_state(self, X, H):
        if H is None:
            H = torch.zeros(X.shape[0], self.out_channels).to(X.device)
        return H

    def _calculate_update_gate(self, g, X, edge_weight, H):
        h = self.conv_z(g, X, edge_weight=edge_weight)
        h = torch.clamp(h, min=-1e6, max=1e6)
        Z = torch.cat((h, H), dim=1)
        Z = self.linear_z(Z)
        return torch.sigmoid(Z)

    def _calculate_reset_gate(self, g, X, edge_weight, H):
        h = self.conv_r(g, X, edge_weight=edge_weight)
        h = torch.clamp(h, min=-1e6, max=1e6)
        R = torch.cat((h, H), dim=1)
        R = self.linear_r(R)
        return torch.sigmoid(R)

    def _calculate_candidate_state(self, g, X, edge_weight, H, R):
        h = self.conv_h(g, X, edge_weight=edge_weight)
        h = torch.clamp(h, min=-1e6, max=1e6)
        H_tilde = torch.cat((h, H * R), dim=1)
        H_tilde = self.linear_h(H_tilde)
        return torch.tanh(H_tilde)

    def _calculate_hidden_state(self, Z, H, H_tilde):
        return Z * H + (1 - Z) * H_tilde

    def _check_fused_inputs(self, g, edge_weight):
        from ....utils.constants import SizeConstants

        for conv in (self.conv_z, self.conv_r, self.conv_h):
            if conv.bias is None or conv.activation is not None:
                raise RuntimeError("the fused TGCN cell needs the three convolutions as the reference builds them "
                                   "(bias, no activation); use TGCN(fused=False)")
        norm = g.get_ndata("norm")
        if norm is None:
            raise KeyError("StaticGraph passed to GCNConv forward pass does not contain 'norm' node data")
        if (len(norm.shape) != SizeConstants.NODE_NORM_SIZE.value or norm.shape[1] != 1
                or norm.shape[0] != g.get_num_nodes()):          # the same check GCNConv.forward makes
            raise ValueError("Node data 'norm' passed to GCNConv should be of shape (num_nodes, 1)")
        if norm.requires_grad or (edge_weight is not None and edge_weight.requires_grad):
            raise RuntimeError("the fused TGCN cell gives no gradient for 'norm' / edge_weight; use TGCN(fused=False)")
        return norm

    def _packed_parameters(self):
        """The cell's parameters in the layout of ``ops_tgcn`` (``[W_z|W_r|W_h]`` ...), packed with differentiable torch
        ops ONCE per BPTT window instead of once per time step: the pack is reused until a parameter changes (in-place
        version counter, storage) or a backward pass has run through it (a hook on the packed weight marks it stale)."""
        from ....ops_tgcn import pack_parameters

        mods = (self.conv_z, self.conv_r, self.conv_h, self.linear_z, self.linear_r, self.linear_h)
        params = [t for m in mods for t in (m.weight, m.bias)]
        key = (torch.is_grad_enabled(),) + tuple((id(t), t._version, t.data_ptr(), t.requires_grad) for t in params)
        cache = self.__dict__.get("_pack_cache")
        if cache is not None and cache[0] == key and not cache[2][0]:
            return cache[1]
        packed = pack_parameters(*mods)
        stale = [False]
        for t in packed:          # any gradient that reaches the pack means a backward pass has run through it
            if t.requires_grad:
                t.register_hook(lambda grad, flag=stale: flag.__setitem__(0, True))
        self.__dict__["_pack_cache"] = (key, packed, stale, {})
        return packed

    def _lowp_parameters(self, packed, dt):
        """The 16-bit GEMM operands of the pack (``ops_tgcn.lowp_parameters``), made once per pack and dtype and kept
        beside it in ``_pack_cache``."""
        from ....ops_tgcn import lowp_parameters

        cache = self.__dict__.get("_pack_cache")
        if cache is None or cache[1] is not packed:
            return lowp_parameters(packed, dt)
        if dt not in cache[3]:
            cache[3][dt] = lowp_parameters(packed, dt)
        return cache[3][dt]

    def _forward_fused(self, g, X, edge_weight, H):
        """The cell as ONE autograd op with a hand-written backward (``ops_tgcn``)."""
        from ....ops_tgcn import tgcn_cell

        norm = self._check_fused_inputs(g, edge_weight)
        packed = self._packed_parameters()
        lowp = None
        if torch.is_autocast_enabled("cuda") and torch.get_autocast_dtype("cuda") in (torch.bfloat16, torch.float16):
            lowp = self._lowp_parameters(packed, torch.get_autocast_dtype("cuda"))
        return tgcn_cell(g, X, H, norm, edge_weight, packed, lowp)

    def _forward_fused_pieces(self, g, X, edge_weight, H):
        """The fused cell of round 1 (``fused="pieces"``): the same kernels, chained by torch autograd piece by piece."""
        from ....ops_gcn import gcn_aggregate
        from ....ops_gru import bias_clamp, gru_reset, gru_update

        norm = self._check_fused_inputs(g, edge_weight)
        hid = self.out_channels
        W = torch.cat((self.conv_z.weight, self.conv_r.weight, self.conv_h.weight), dim=1)
        b = torch.cat((self.conv_z.bias, self.conv_r.bias, self.conv_h.bias))
        # bias add + clamp(+-1e6) in one in-place pass over the [N, 3H] aggregation output
        h = bias_clamp(gcn_aggregate(g, torch.mm(X, W), norm, edge_weight), b, -1e6, 1e6)
        hz, hr, hh = h.split(hid, dim=1)          # split: the backward is one concatenation, not three zero-filled slices

        def gate(linear, a, c):      # linear(cat(a, c)) without materialising the concatenation: two GEMMs
            return torch.addmm(torch.addmm(linear.bias, a, linear.weight[:, :hid].t()), c, linear.weight[:, hid:].t())

        pz = gate(self.linear_z, hz, H)
        pr = gate(self.linear_r, hr, H)
        ph = gate(self.linear_h, hh, gru_reset(pr, H))          # H * sigmoid(pr)
        return gru_update(pz, ph, H)                            # Z * H + (1 - Z) * tanh(ph)

    def _can_fuse(self, g, edge_weight) -> bool:
        convs = (self.conv_z, self.conv_r, self.conv_h)
        norm = g.get_ndata("norm") if hasattr(g, "get_ndata") else None
        return (all(type(c) is GCNConv and c.activation is None and c.bias is not None for c in convs)
                and not hasattr(g, "num_local_nodes") and norm is not None and not norm.requires_grad
                and (not torch.is_autocast_enabled("cuda")         # the one-op cell has an fp32 and a bf16 / fp16 form
                     or torch.get_autocast_dtype("cuda") in (torch.bfloat16, torch.float16))
                and (edge_weight is None or not edge_weight.requires_grad))

    def forward(self, g, X, edge_weight=None, H=None):
        if self.fused or (self.fused is None and self._can_fuse(g, edge_weight)):
            if H is None:      # allocated on the device directly: no H2D copy, CUDA-graph capturable
                # under autocast the hidden state is fp32 (X is 16-bit when a model's own Linear feeds the cell)
                dtype = torch.float32 if torch.is_autocast_enabled("cuda") else X.dtype
                H = torch.zeros(X.shape[0], self.out_channels, device=X.device, dtype=dtype)
            if self.fused == "pieces":
                return self._forward_fused_pieces(g, X, edge_weight, H)
            return self._forward_fused(g, X, edge_weight, H)
        H = self._set_hidden_state(X, H)
        Z = self._calculate_update_gate(g, X, edge_weight, H)
        R = self._calculate_reset_gate(g, X, edge_weight, H)
        H_tilde = self._calculate_candidate_state(g, X, edge_weight, H, R)
        return self._calculate_hidden_state(Z, H, H_tilde)
