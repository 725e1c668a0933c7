"""Reference multi-head GATConv for the tests: the oracle's ``GATConv`` (any heads, concat) and PyG 2.5.2's ``concat=False``
written with the oracle's own helpers (gat_conv.py: per-head softmax and aggregation as for concat, then ``out.mean(dim=1)``,
then ``+ bias``).  Parameter names, order, shapes and init are PyG's: ``lin.weight``, ``att_src``, ``att_dst``, ``bias``, so
``state_dict()`` loads into ``deformcontact_b200.GATConv(..., concat=False)`` unchanged."""
import torch
import torch.nn as nn
import torch.nn.functional as F

import oracle
from oracle import convs


class GATConvMean(nn.Module):
    """PyG ``GATConv(in, out, heads=H, concat=False)``: the mean over the H heads, + ``bias [out]``."""

    def __init__(self, in_channels, out_channels, heads=1, negative_slope=0.2, bias=True):
        super().__init__()
        init = oracle.GATConv(in_channels, out_channels, heads=heads, negative_slope=negative_slope, bias=False)
        self.lin, self.att_src, self.att_dst = init.lin, init.att_src, init.att_dst
        self.bias = nn.Parameter(torch.zeros(out_channels)) if bias else None
        self.in_channels, self.out_channels, self.heads, self.negative_slope = in_channels, out_channels, heads, negative_slope
        self.concat = False

    def forward(self, x, edge_index):
        n, H, C = x.shape[0], self.heads, self.out_channels
        xs = self.lin(x).view(n, H, C)
        a_src = (xs * self.att_src).sum(-1)
        a_dst = (xs * self.att_dst).sum(-1)
        edge_index = convs.add_self_loops(convs.remove_self_loops(edge_index), n)
        row, col = edge_index[0], edge_index[1]
        alpha = convs.segment_softmax(F.leaky_relu(a_src[row] + a_dst[col], self.negative_slope), col, n)
        out = convs._scatter_sum(alpha.unsqueeze(-1) * xs.index_select(0, row), col, n).mean(dim=1)
        return out + self.bias if self.bias is not None else out


def gat_reference(in_channels, out_channels, heads=1, concat=True, negative_slope=0.2, bias=True):
    """The oracle's GATConv for ``concat=True``, ``GATConvMean`` for ``concat=False``; both carry ``.concat``."""
    if not concat:
        return GATConvMean(in_channels, out_channels, heads=heads, negative_slope=negative_slope, bias=bias)
    layer = oracle.GATConv(in_channels, out_channels, heads=heads, negative_slope=negative_slope, bias=bias)
    layer.concat = True
    return layer
