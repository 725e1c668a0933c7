"""Drop-in message-passing layers: ``TAGConv`` / ``GCNConv`` / ``GATConv`` (+ ``MPNNLayer``).

Same constructor signature ``(in_channels, out_channels)``, call ``layer(x, edge_index)`` and
state-dict keys as torch_geometric 2.5.2, so they slot into the reference's
``GraphNet.__init__`` / ``forward`` (models/model.py:39-50, 69-78) and load its checkpoints
(train.py:125, eval.py:36,89).  Forward and backward run entirely in libdcb200 (hand-written
sm_100a CUDA reached through the C ABI); every layer is ONE registered custom op with a registered
autograd formula (``torch.ops.dcb200.{tag_conv, gcn_conv, gat_conv / gat_conv_heads, mpnn_layer}``, torch_ops.py) — the
modules below only hold the parameters and call the op.

``edge_index`` may be the usual ``int64 [2, E]`` tensor (the CSR pair is built once per tensor
and cached) or a prebuilt ``ops.GraphCSR`` (adopted into that cache under its own ``edge_index``).

``TAGConv`` / ``GCNConv`` take PyG's ``edge_weight`` (fp32 CUDA ``[E]``, in the order of ``edge_index``, or of the tensor a
prebuilt ``GraphCSR`` was built from).  ``GraphNet`` / ``CapturedTrainStep`` pass none (neither does the reference), and
``Batch`` does not collate per-edge weights: concatenate them in the batch's edge order.
"""
import math

import os

import torch
import torch.nn as nn

from . import ops
from . import torch_ops  # noqa: F401  (registers torch.ops.dcb200.*)


def _kaiming_uniform_linear_(w):
    bound = 1.0 / math.sqrt(w.size(-1)) if w.size(-1) > 0 else 0.0
    with torch.no_grad():
        w.uniform_(-bound, bound)


def _glorot_(w):
    a = math.sqrt(6.0 / (w.size(-2) + w.size(-1)))
    with torch.no_grad():
        w.uniform_(-a, a)


class _Lin(nn.Module):
    """Holds ``weight [out, in]`` under PyG's ``lins.k.weight`` / ``lin.weight`` key."""

    def __init__(self, i, o, init="kaiming"):
        super().__init__()
        self.weight = nn.Parameter(torch.empty(o, i))
        (_glorot_ if init == "glorot" else _kaiming_uniform_linear_)(self.weight)


def _edge_tensor(edge_index):
    """The tensor the custom ops take: ``edge_index`` itself, or — for a prebuilt ``ops.GraphCSR`` — the tensor it was built
    from, after adopting the structure into the cache the ops look it up in."""
    if isinstance(edge_index, ops.GraphCSR):
        return ops.adopt_csr(edge_index)
    return edge_index


def _edge_weight(edge_weight, edge_index):
    """``edge_weight`` checked against the edges it weights: None, or fp32 CUDA [E] in the order of ``edge_index`` (of the tensor a
    prebuilt ``ops.GraphCSR`` was built from).  ``relu`` / ``ptr`` used to be the third and fourth arguments: a ``bool`` here is a
    positional ``relu`` and is refused rather than taken as a weight."""
    if edge_weight is None:
        return None
    if isinstance(edge_weight, bool) or not isinstance(edge_weight, torch.Tensor):
        raise TypeError(f"edge_weight must be a float32 tensor [E] or None, got {type(edge_weight).__name__} "
                        "(pass relu and ptr by keyword)")
    if edge_weight.dtype != torch.float32:
        raise ops._abi.DcError(f"edge_weight: expected dtype torch.float32, got {edge_weight.dtype}")
    E = edge_index.E if isinstance(edge_index, ops.GraphCSR) else edge_index.shape[1]
    if edge_weight.dim() != 1 or edge_weight.shape[0] != E:
        raise ops._abi.DcError(f"edge_weight: expected [{E}] (one weight per edge), got {tuple(edge_weight.shape)}")
    if not edge_weight.is_cuda:
        raise ops._abi.DcError("edge_weight: expected a CUDA tensor (libdcb200 has no CPU path)")
    dev = edge_index.rowptr.device if isinstance(edge_index, ops.GraphCSR) else edge_index.device
    if edge_weight.device != dev:
        raise ops._abi.DcError(f"edge_weight is on {edge_weight.device}, edge_index on {dev}")
    return edge_weight


def _pad4(x, weights, chain=False):
    """Zero-pad the feature axis of ``x`` and the input axis of ``weights`` to a multiple of 4 floats (16-byte rows) so the
    vector hop kernels and the tensor-core GEMM take layers whose input width is not one (21 / 25 in everyday.json).
    The padding columns are exact zeros end to end; ``F.pad`` keeps autograd (the gradients are sliced back)."""
    pad = (-x.shape[1]) % 4
    if chain and x.shape[1] < 32 and PAD_CHAIN_WIDTH:
        pad = 32 - x.shape[1]      # one 128-byte slice: the K hops of the layer run as ONE chain launch (needs F % 32 == 0)
    if pad == 0 or not PAD_INPUT_WIDTH:
        return x, weights
    return nn.functional.pad(x, (0, pad)), [nn.functional.pad(w, (0, pad)) for w in weights]


PAD_INPUT_WIDTH = True
PAD_CHAIN_WIDTH = os.environ.get("DCB200_PAD_CHAIN", "1") == "1"   # TAGConv inputs narrower than 32 (21 / 25): pad to 32 instead of 24 / 28


# ------------------------------------------------------------------------------- TAGConv
class TAGConv(nn.Module):
    """PyG ``TAGConv(in, out, K=3, bias=True, normalize=True)``; keys ``lins.{0..K}.weight``, ``bias``.
    out = act( sum_k A_hat^k X W_k^T + b ): K hops in one chain launch (K1) + one multi-segment GEMM with bias / ReLU
    epilogue (K2); backward dH_k = dOut W_k, dW_k = dOut^T H_k, db = colsum(dOut), then the K transposed hops as one chain
    accumulating in place (``torch.ops.dcb200.tag_conv`` / ``tag_conv_backward``).

    ``layer(x, edge_index, edge_weight=None)`` as in PyG: ``edge_weight`` fp32 CUDA [E] in ``edge_index`` order.  With
    ``normalize`` A_hat is PyG's weighted ``gcn_norm(add_self_loops=False)``, computed on the device every call; without, the
    weights themselves.  ``torch.ops.dcb200.tag_conv_weighted``: the same hops on the weighted norms, and dL/dedge_weight (when
    the weights require grad) from one SDDMM over the saved hops and the normalisation backward.  Where incoming weights sum to
    exactly 0 the degree gradient is 0 (PyG's autograd gives NaN).  SparseTensor adjacency is not supported."""

    def __init__(self, in_channels, out_channels, K=3, bias=True, normalize=True, precision=ops.GEMM_AUTO):
        super().__init__()
        self.in_channels, self.out_channels, self.K, self.normalize = in_channels, out_channels, K, normalize
        self.lins = nn.ModuleList([_Lin(in_channels, out_channels) for _ in range(K + 1)])
        self.bias = nn.Parameter(torch.zeros(out_channels)) if bias else None
        self.precision = precision

    def forward(self, x, edge_index, edge_weight=None, relu=False, ptr=None):
        edge_weight = _edge_weight(edge_weight, edge_index)
        x, ws = _pad4(x, [l.weight for l in self.lins], chain=True)
        if edge_weight is not None:
            return torch.ops.dcb200.tag_conv_weighted(x, _edge_tensor(edge_index), edge_weight, ws, self.bias, relu, self.normalize,
                                                      self.precision, ptr)[0]
        return torch.ops.dcb200.tag_conv(x, _edge_tensor(edge_index), ws, self.bias, relu, self.normalize, self.precision, ptr)[0]


def layer_stack(layers, x, edge_index, relu=True, ptr=None, between=None, edge_weight=None):
    """``for conv in layers: x = act(conv(x, edge_index, edge_weight))`` (models/model.py:69-78) for TAGConv / GCNConv layers on
    ONE graph.  A relabelled large graph (one cloud of >= 32768 points from ``knn_graph`` / ``radius_graph``) is entered once and
    left once: its features stay in the structure's node order from layer to layer (bit-identical to the plain loop, which
    permutes in and out of every layer; relabelling keeps the edge order, so ``edge_weight`` applies unchanged).  ``between``:
    optional callable applied after every layer (dropout)."""
    mode = {"TAGConv": "tag", "GCNConv": "gcn"}.get(type(layers[0]).__name__) if len(layers) else None
    same = mode is not None and all(type(l) is type(layers[0]) for l in layers)
    if mode == "tag" and same and not all(getattr(l, "normalize", True) for l in layers):
        same = False
    g = None
    if same and not isinstance(edge_index, ops.GraphCSR):
        x, edge_index, g = ops.stack_enter(x, edge_index, mode, ptr)
    kw = {} if edge_weight is None else {"edge_weight": edge_weight}
    for conv in layers:
        x = conv(x, edge_index, relu=relu, ptr=ptr, **kw)
        if between is not None:
            x = between(x)
    return ops.stack_exit(x, g)


# ------------------------------------------------------------------------------- GCNConv
class GCNConv(nn.Module):
    """PyG ``GCNConv(in, out, improved=False)`` with its other defaults; keys ``lin.weight``, ``bias``.

    ``layer(x, edge_index, edge_weight=None)`` as in PyG: ``edge_weight`` fp32 CUDA [E] in ``edge_index`` order.  Weights or
    ``improved`` run ``torch.ops.dcb200.gcn_conv_weighted``: PyG's weighted ``gcn_norm`` with ``add_remaining_self_loops``
    computed on the device every call — a node's loop takes the weight of its LAST self-loop edge (edge order), else
    ``fill_value`` = 2 if ``improved`` else 1 — and, when the weights require grad, dL/dedge_weight from one SDDMM and the
    normalisation backward.  The loop's gradient goes to the edge that supplied its weight; superseded duplicate loops get 0
    (PyG's ``index_put`` autograd also credits them), and where the weights into a node sum to exactly 0 the degree gradient
    is 0 (PyG: NaN).  ``cached``, ``add_self_loops=False``, ``normalize=False`` and SparseTensor adjacency are not supported:
    the first three raise."""

    def __init__(self, in_channels, out_channels, bias=True, precision=ops.GEMM_AUTO, *, improved=False, cached=False,
                 add_self_loops=True, normalize=True):
        super().__init__()
        if cached or not add_self_loops or not normalize:
            raise NotImplementedError("GCNConv: cached, add_self_loops=False and normalize=False are not supported")
        self.in_channels, self.out_channels, self.improved = in_channels, out_channels, bool(improved)
        self.lin = _Lin(in_channels, out_channels, init="glorot")
        self.bias = nn.Parameter(torch.zeros(out_channels)) if bias else None
        self.precision = precision

    def forward(self, x, edge_index, edge_weight=None, relu=False, ptr=None):
        edge_weight = _edge_weight(edge_weight, edge_index)
        if edge_weight is None and not self.improved:
            return torch.ops.dcb200.gcn_conv(x, _edge_tensor(edge_index), self.lin.weight, self.bias, relu, self.precision, ptr)
        if edge_weight is None:
            E = edge_index.E if isinstance(edge_index, ops.GraphCSR) else edge_index.shape[1]
            edge_weight = torch.ones(E, dtype=torch.float32, device=x.device)
        return torch.ops.dcb200.gcn_conv_weighted(x, _edge_tensor(edge_index), edge_weight, self.lin.weight, self.bias, relu,
                                                  2.0 if self.improved else 1.0, self.precision, ptr)[0]


# ------------------------------------------------------------------------------- GATConv
class GATConv(nn.Module):
    """PyG 2.5.x ``GATConv(in, out, heads=1, concat=True, negative_slope=0.2, bias=True)`` with ``add_self_loops=True`` and
    ``dropout=0``; keys ``lin.weight [H*C, in]``, ``att_src`` / ``att_dst [1, H, C]``, ``bias [H*C]`` (concat) or ``[C]`` (mean).

    ``heads == 1`` runs ``torch.ops.dcb200.gat_conv`` (scores, softmax, then the K1 aggregation).  ``heads > 1`` runs
    ``torch.ops.dcb200.gat_conv_heads``: per-head softmax and aggregation in one launch with the concat / mean epilogue
    (``dc_gat_aggregate``), backward by receiver then by source (``dc_gat_bwd_edge_heads``, ``dc_gat_scatter_heads``).
    Attention dropout, ``add_self_loops=False``, ``fill_value`` and ``edge_dim`` are not supported and raise; the call takes no
    ``edge_attr``.

    ``layer(x, edge_index, return_attention_weights=...)`` as in PyG 2.5.2:

    - ``None`` (the default): the output tensor.
    - any ``bool``, ``False`` included (PyG tests ``isinstance(..., bool)``): ``(out, (edge_index_sl, alpha))``.
      ``edge_index_sl`` int64 ``[2, E_nl + N]`` is ``add_self_loops(remove_self_loops(edge_index), N)``: the edges that are not
      self loops in their order (duplicates kept), then one loop per node, in the node labels of ``edge_index`` (of the tensor a
      prebuilt ``GraphCSR`` was built from).  It is built once per structure and shared by later calls: do not write to it.
      ``alpha`` fp32 ``[E_nl + N, H]`` (the head axis kept for H = 1) holds the coefficients the aggregation used, row for row,
      and is differentiable: a loss on ``alpha`` (an entropy or sparsity regulariser) reaches ``x`` and every parameter.
      ``relu`` applies to ``out`` only.  Any other value raises ``TypeError``.

    With attention weights every ``heads`` runs ``gat_conv_heads``, which keeps alpha per head; the gradient that reaches alpha
    enters its receiver pass (``dc_gat_bwd_edge_heads_ext``).  For H = 1 ``out`` is therefore within rounding of, not
    bit-identical to, the call without.  The first call on a structure reads the edge count back to the host once."""

    def __init__(self, in_channels, out_channels, heads=1, concat=True, negative_slope=0.2, bias=True, precision=ops.GEMM_AUTO, *,
                 dropout=0.0, add_self_loops=True, edge_dim=None, fill_value="mean"):
        super().__init__()
        if heads < 1:
            raise ValueError(f"GATConv: heads must be >= 1, got {heads}")
        if dropout != 0.0 or not add_self_loops or edge_dim is not None or fill_value != "mean":
            raise NotImplementedError("GATConv: attention dropout, add_self_loops=False, fill_value and edge_dim are not supported")
        self.in_channels, self.out_channels, self.heads, self.negative_slope = in_channels, out_channels, heads, negative_slope
        self.concat = concat
        self.lin = _Lin(in_channels, heads * out_channels, init="glorot")
        self.att_src = nn.Parameter(torch.empty(1, heads, out_channels))
        self.att_dst = nn.Parameter(torch.empty(1, heads, out_channels))
        _glorot_(self.att_src)
        _glorot_(self.att_dst)
        self.bias = nn.Parameter(torch.zeros(heads * out_channels if concat else out_channels)) if bias else None
        self.precision = precision

    def forward(self, x, edge_index, relu=False, ptr=None, *, return_attention_weights=None):
        if return_attention_weights is not None and not isinstance(return_attention_weights, bool):
            raise TypeError("return_attention_weights must be None or a bool, got "
                            f"{type(return_attention_weights).__name__}")
        ei = _edge_tensor(edge_index)
        if return_attention_weights is None and self.heads == 1:   # the mean over one head is that head: concat = mean
            return torch.ops.dcb200.gat_conv(x, ei, self.lin.weight, self.att_src, self.att_dst, self.bias,
                                             float(self.negative_slope), relu, self.precision, ptr)[0]
        res = torch.ops.dcb200.gat_conv_heads(x, ei, self.lin.weight, self.att_src, self.att_dst, self.bias,
                                              float(self.negative_slope), self.heads, bool(self.concat), relu, self.precision, ptr)
        if return_attention_weights is None:
            return res[0]
        g = ops.graph_csr(ei, x.shape[0], "gat", list(ptr) if ptr is not None else None)
        keep, edge_index_sl = g.attention_edges()
        return res[0], (edge_index_sl, ops.attention_weights(res[4], res[5], keep, g.E))


# ------------------------------------------------------------------------------- MPNN (A9 extension)
class MPNNLayer(nn.Module):
    """``MPNNLayer(in, out)``; keys ``edge_mlp.{0,2}.{weight,bias}``, ``node_mlp.{0,2}.{weight,bias}``
    (``nn.Sequential(Linear, ReLU, Linear)`` each).  Residual when ``in == out``.  Needs ``out % 4 == 0``."""

    def __init__(self, in_channels, out_channels, precision=ops.GEMM_AUTO):
        super().__init__()
        if out_channels % 4:
            raise NotImplementedError("MPNNLayer: out_channels must be a multiple of 4")
        self.in_channels, self.out_channels, self.precision = in_channels, out_channels, precision
        self.edge_mlp = nn.Sequential(nn.Linear(2 * in_channels, out_channels), nn.ReLU(), nn.Linear(out_channels, out_channels))
        self.node_mlp = nn.Sequential(nn.Linear(in_channels + out_channels, out_channels), nn.ReLU(),
                                      nn.Linear(out_channels, out_channels))

    def forward(self, x, edge_index, relu=False, ptr=None):
        out = torch.ops.dcb200.mpnn_layer(x, _edge_tensor(edge_index), self.edge_mlp[0].weight, self.edge_mlp[0].bias,
                                          self.edge_mlp[2].weight, self.edge_mlp[2].bias, self.node_mlp[0].weight,
                                          self.node_mlp[0].bias, self.node_mlp[2].weight, self.node_mlp[2].bias,
                                          self.in_channels == self.out_channels, self.precision, ptr)[0]
        return torch.relu(out) if relu else out
