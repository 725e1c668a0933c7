"""Reference GATConv with PyG 2.5.2's ``return_attention_weights`` for the tests, written with the oracle's helpers
(``convs.add_self_loops``, ``remove_self_loops``, ``segment_softmax``): ``None`` returns ``out``; any ``bool`` (``False``
included) returns ``(out, (edge_index_sl, alpha))`` with ``edge_index_sl = add_self_loops(remove_self_loops(edge_index), N)``
and ``alpha [E_nl + N, H]`` in its order.  Concat or the mean over heads, + bias.  Parameter names, order, shapes and init are
PyG's (those of ``tests/gat_reference.py``), so ``state_dict()`` loads into and from ``deformcontact_b200.GATConv``."""
import torch.nn as nn
import torch.nn.functional as F

from oracle import convs
from gat_reference import gat_reference


class GATConvAttention(nn.Module):
    def __init__(self, in_channels, out_channels, heads=1, concat=True, negative_slope=0.2, bias=True):
        super().__init__()
        init = gat_reference(in_channels, out_channels, heads=heads, concat=concat, negative_slope=negative_slope, bias=bias)
        self.lin, self.att_src, self.att_dst, self.bias = init.lin, init.att_src, init.att_dst, init.bias
        self.in_channels, self.out_channels, self.heads, self.negative_slope = in_channels, out_channels, heads, negative_slope
        self.concat = concat

    def forward(self, x, edge_index, return_attention_weights=None):
        n, H, C = x.shape[0], self.heads, self.out_channels
        xs = self.lin(x).view(n, H, C)
        a_src = (xs * self.att_src).sum(-1)
        a_dst = (xs * self.att_dst).sum(-1)
        edge_index = convs.add_self_loops(convs.remove_self_loops(edge_index), n)
        row, col = edge_index[0], edge_index[1]
        alpha = convs.segment_softmax(F.leaky_relu(a_src[row] + a_dst[col], self.negative_slope), col, n)
        out = convs._scatter_sum(alpha.unsqueeze(-1) * xs.index_select(0, row), col, n)
        out = out.reshape(n, H * C) if self.concat else out.mean(dim=1)
        if self.bias is not None:
            out = out + self.bias
        if isinstance(return_attention_weights, bool):
            return out, (edge_index, alpha)
        return out
