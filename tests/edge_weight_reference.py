"""Reference TAGConv / GCNConv with PyG's ``edge_weight`` for the tests, written with the oracle's own helpers (as
tests/gat_reference.py is): PyG 2.5.2's weighted ``gcn_norm`` (nn/conv/gcn_conv.py) with ``add_remaining_self_loops``
(utils/loop.py) for GCNConv, then the oracle's ``propagate``.

Two choices where PyG's autograd is not what the library computes, both on purpose:
- a node's appended loop takes the weight of its LAST self-loop edge (edge order; PyG's ``loop_attr[idx] = edge_attr[mask]``
  on the CPU, where the last write wins), and its gradient goes to that edge alone (PyG's ``index_put`` autograd also credits
  the superseded loops);
- where the weights into a node sum to exactly 0, dis = 0 and the degree gradient is 0 (PyG: NaN).
Parameter names, order, shapes and init are PyG's, so ``state_dict()`` loads into ``deformcontact_b200``'s layers."""
import torch

import oracle
from oracle import convs


def last_loop_edge(edge_index, n):
    """int64 [n]: the largest edge id e with src_e == dst_e == node, else -1."""
    loops = torch.nonzero(edge_index[0] == edge_index[1]).flatten()
    last = torch.full((n,), -1, dtype=torch.long, device=edge_index.device)
    return last.scatter_reduce(0, edge_index[0, loops], loops, reduce="amax", include_self=True)


def gcn_norm_weighted(edge_index, edge_weight, n, add_self_loops=False, fill_value=1.0):
    """PyG ``gcn_norm(edge_index, edge_weight, n, improved=fill_value == 2, add_self_loops)`` -> (edge_index, norm)."""
    w = edge_weight
    if add_self_loops:
        keep = edge_index[0] != edge_index[1]
        last = last_loop_edge(edge_index, n)
        loop_w = torch.cat([w, w.new_full((1,), fill_value)])[torch.where(last >= 0, last, w.shape[0])]   # index E: fill_value
        edge_index = convs.add_self_loops(edge_index[:, keep], n)
        w = torch.cat([w[keep], loop_w])
    row, col = edge_index[0], edge_index[1]
    deg = convs._scatter_sum(w, col, n)
    zero = deg == 0
    dis = torch.where(zero, torch.zeros_like(deg), torch.where(zero, torch.ones_like(deg), deg).pow(-0.5))
    return edge_index, dis[row] * w * dis[col]


class TAGConvWeighted(oracle.TAGConv):
    """``oracle.TAGConv`` called as ``conv(x, edge_index, edge_weight)``."""

    def forward(self, x, edge_index, edge_weight):
        n = x.shape[0]
        if self.normalize:
            edge_index, w = gcn_norm_weighted(edge_index, edge_weight, n, False)
        else:
            w = edge_weight
        out = self.lins[0](x)
        for lin in self.lins[1:]:
            x = convs.propagate(x, edge_index, w, n)
            out = out + lin(x)
        return out + self.bias if self.bias is not None else out


class GCNConvWeighted(oracle.GCNConv):
    """``oracle.GCNConv`` with ``improved`` and ``conv(x, edge_index, edge_weight)``."""

    def __init__(self, in_channels, out_channels, improved=False, bias=True):
        super().__init__(in_channels, out_channels, bias=bias)
        self.improved = improved

    def forward(self, x, edge_index, edge_weight):
        n = x.shape[0]
        edge_index, w = gcn_norm_weighted(edge_index, edge_weight, n, True, 2.0 if self.improved else 1.0)
        out = convs.propagate(self.lin(x), edge_index, w, n)
        return out + self.bias if self.bias is not None else out


def dense_adjacency_fp64(edge_index, edge_weight, n, add_self_loops=False, fill_value=1.0, normalize=True):
    """Independent dense fp64 formulation: A[i, j] = sum of the weights of the edges j -> i (for GCN: non-loop edges, and
    the diagonal = the last loop's weight or fill_value), normalised by D^-1/2 A D^-1/2 with D = row sums."""
    w = edge_weight.double()
    A = torch.zeros(n, n, dtype=torch.float64)
    if add_self_loops:
        keep = edge_index[0] != edge_index[1]
        A = A.index_put((edge_index[1, keep], edge_index[0, keep]), w[keep], accumulate=True)
        last = last_loop_edge(edge_index, n)
        diag = torch.cat([w, w.new_full((1,), fill_value)])[torch.where(last >= 0, last, w.shape[0])]
        A = A + torch.diag(diag)
    else:
        A = A.index_put((edge_index[1], edge_index[0]), w, accumulate=True)
    if not normalize:
        return A
    deg = A.sum(1)
    dis = torch.where(deg == 0, torch.zeros_like(deg), torch.where(deg == 0, torch.ones_like(deg), deg).pow(-0.5))
    return dis[:, None] * A * dis[None, :]
