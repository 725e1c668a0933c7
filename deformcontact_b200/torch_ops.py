"""``torch.ops.dcb200.*`` — the kernels as registered PyTorch custom ops (SURVEY.md 8b, "Torch op layer").

Thin layer over ``ops.py`` (which is itself a thin layer over the C ABI): every op has a CUDA
implementation that enqueues libdcb200 kernels on the current stream, a fake (meta) implementation so
it traces under ``torch.compile`` / CUDA-graph capture tooling, and — for the layer ops — a registered
autograd formula whose backward is again a ``dcb200`` op.  This file holds the ONLY implementation of the
four layers' forward / backward; the ``nn.Module``s in ``layers.py`` call these ops and nothing else.

    csr_build, propagate, linear, knn_table, radius_table, knn_graph, radius_graph,
    tag_conv(+_backward), gcn_conv(+_backward), tag_conv_weighted(+_backward), gcn_conv_weighted(+_backward),
    gat_conv(+_backward), gat_conv_heads(+_backward), mpnn_layer(+_backward)
"""
from typing import List, Optional, Tuple

import torch
from torch import Tensor

from . import ops

_lib = torch.library


def _csr(edge_index, n, mode, ptr):
    return ops.graph_csr(edge_index, n, mode, list(ptr) if ptr is not None else None)


# ----------------------------------------------------------------------------------- primitives
@_lib.custom_op("dcb200::csr_build", mutates_args=())
def csr_build(edge_index: Tensor, num_nodes: int, group_by: int, drop_self_loops: bool) -> Tuple[Tensor, Tensor, Tensor]:
    return ops.csr_build(edge_index, num_nodes, group_by, drop_self_loops)


@csr_build.register_fake
def _(edge_index, num_nodes, group_by, drop_self_loops):
    E = edge_index.shape[1]
    i32 = dict(dtype=torch.int32, device=edge_index.device)
    return torch.empty(num_nodes + 1, **i32), torch.empty(E, **i32), torch.empty(E, **i32)


@_lib.custom_op("dcb200::propagate", mutates_args=())
def propagate(h: Tensor, edge_index: Tensor, mode: str, transpose: bool, add: Optional[Tensor], bias: Optional[Tensor],
              relu: bool, ptr: Optional[List[int]]) -> Tensor:
    """One hop: act(add + A_hat h + bias) (A_hat^T if transpose); A_hat per mode 'tag' | 'gcn' | 'plain'."""
    return _csr(edge_index, h.shape[0], mode, ptr).propagate(h.contiguous(), transpose=transpose, add=add, bias=bias, relu=relu)


@propagate.register_fake
def _(h, edge_index, mode, transpose, add, bias, relu, ptr):
    return torch.empty_like(h, memory_format=torch.contiguous_format)


@_lib.custom_op("dcb200::linear", mutates_args=())
def linear(x: Tensor, weight: Tensor, bias: Optional[Tensor], relu: bool) -> Tensor:
    """act(x W^T + b) on the tcgen05 3xTF32 / fp32 GEMM (dc_gemm)."""
    return ops.gemm([(x.contiguous(), weight)], x.shape[0], weight.shape[0], False, True, bias=bias, relu=relu)


@linear.register_fake
def _(x, weight, bias, relu):
    return x.new_empty((x.shape[0], weight.shape[0]))


@_lib.custom_op("dcb200::knn_table", mutates_args=())
def knn_table(pos: Tensor, k: int, ptr: Optional[Tensor], loop: bool) -> Tensor:
    return ops.knn_table(pos, k, ptr=ptr, loop=loop)


@knn_table.register_fake
def _(pos, k, ptr, loop):
    return torch.empty((pos.shape[0], k + (0 if loop else 1)), dtype=torch.int32, device=pos.device)


@_lib.custom_op("dcb200::radius_table", mutates_args=())
def radius_table(pos: Tensor, r: float, ptr: Optional[Tensor], loop: bool, max_num_neighbors: int) -> Tuple[Tensor, Tensor]:
    return ops.radius_table(pos, r, ptr=ptr, loop=loop, max_num_neighbors=max_num_neighbors)


@radius_table.register_fake
def _(pos, r, ptr, loop, max_num_neighbors):
    n = pos.shape[0]
    return (torch.empty((n, max_num_neighbors + (0 if loop else 1)), dtype=torch.int32, device=pos.device),
            torch.empty(n, dtype=torch.int32, device=pos.device))


# ----------------------------------------------------------------------------------- TAGConv
@_lib.custom_op("dcb200::tag_conv", mutates_args=())
def tag_conv(x: Tensor, edge_index: Tensor, weights: List[Tensor], bias: Optional[Tensor], relu: bool, normalize: bool,
             precision: int, ptr: Optional[List[int]]) -> Tuple[Tensor, Tensor]:
    """-> (out [N, Fo], hops [N, K*Fi]) ; hops = [A x | A^2 x | ...] is kept for the backward."""
    return _tag_forward(_csr(edge_index, x.shape[0], "tag" if normalize else "plain", ptr), x, weights, bias, relu, precision)


def _tag_forward(g, x, weights, bias, relu, precision):
    x = x.contiguous()
    N, Fi = x.shape
    K = len(weights) - 1
    buf = torch.empty((N, max(K, 1) * Fi), dtype=x.dtype, device=x.device)
    hs = [g.to_internal(x)]   # a relabelled large graph (ops.REORDER) runs the whole layer in its own node order
    for k in range(K):
        hs.append(buf[:, k * Fi:(k + 1) * Fi])
    if K:
        ops.propagate_chain(g, [(hs[k], None, hs[k + 1]) for k in range(K)], internal=True)   # h_{k+1} = A_hat h_k (one launch, K1 v9)
    out = ops.gemm([(h, w) for h, w in zip(hs, weights)], N, weights[0].shape[0], False, True, bias=bias, relu=relu,
                   precision=precision)
    return g.from_internal(out), buf


@tag_conv.register_fake
def _(x, edge_index, weights, bias, relu, normalize, precision, ptr):
    K = len(weights) - 1
    return x.new_empty((x.shape[0], weights[0].shape[0])), x.new_empty((x.shape[0], max(K, 1) * x.shape[1]))


@_lib.custom_op("dcb200::tag_conv_backward", mutates_args=())
def tag_conv_backward(dout: Tensor, out: Tensor, x: Tensor, hops: Tensor, edge_index: Tensor, weights: List[Tensor],
                      relu: bool, normalize: bool, precision: int, ptr: Optional[List[int]], need_dx: bool, need_db: bool,
                      need_dw: bool) -> Tuple[Tensor, Tensor, Tensor]:
    """-> (dx, dbias, dW stacked [K+1, Fo, Fi]); empty tensors for gradients that are not needed."""
    g = _csr(edge_index, x.shape[0], "tag" if normalize else "plain", ptr)
    dx, db, dws, _, _ = _tag_backward_impl(g, dout, out, x, hops, weights, relu, precision, need_dx, need_db, need_dw)
    return dx, db, dws


def _tag_backward_impl(g, dout, out, x, hops, weights, relu, precision, need_dx, need_db, need_dw, need_chain=False):
    """-> (dx, dbias, dWs, dhs, hs): dhs[k] = G_k = dL/dH_k (the totals the transposed chain leaves, structure order) for
    k >= 1 when ``need_chain`` or ``need_dx`` (and k = 0 with ``need_dx``), hs = [x, A x, ...] in structure order."""
    dout, db = ops.relu_bwd_db(out, dout.contiguous(), relu, need_db)   # ReLU backward + bias gradient in one pass
    dout = g.to_internal(dout)      # the saved hops are in the structure's node order
    N, Fo = dout.shape
    Fi = x.shape[1]
    K = len(weights) - 1
    hs = [g.to_internal(x.contiguous())] + [hops[:, k * Fi:(k + 1) * Fi] for k in range(K)]
    if need_dw:
        dws = torch.empty((K + 1, Fo, Fi), dtype=dout.dtype, device=dout.device)
        for k, h in enumerate(hs):
            ops.gemm([(dout, h)], Fo, Fi, True, False, out=dws[k], precision=precision)
    else:
        dws = dout.new_empty(0)
    db = db if need_db else dout.new_empty(0)
    dhs = None
    if need_dx or need_chain:
        lo = 0 if need_dx else 1        # G_0 = dx is only needed for dx
        if ops.K1_CHAIN >= 2 and K > 0:
            # all dH_k = dOut W_k first — ONE batched tensor-core launch over the K + 1 weights where the shapes allow it (same
            # tiles and arithmetic as K + 1 dc_gemm calls, a quarter of the launches / pipeline ramps) — then the transposed hops as
            # one chain, accumulating in place: dH_{k-1} += A_hat^T g_k
            dhs = [None] * lo
            if (precision != ops.GEMM_FP32 and ops.FORCE_GEMM_PRECISION != ops.GEMM_FP32 and Fi % 4 == 0 and Fo % 4 == 0
                    and float(N) * Fo * Fi >= 1.0e8 and all(w.stride(0) % 4 == 0 and w.data_ptr() % 16 == 0 for w in weights)):
                dhs += [torch.empty((N, Fi), dtype=dout.dtype, device=dout.device) for _ in range(lo, K + 1)]
                ops.gemm_batched([(dout, weights[k], dhs[k]) for k in range(lo, K + 1)], trans_a=False, trans_b=False)
            else:
                dhs += [ops.gemm([(dout, weights[k])], N, Fi, False, False, precision=precision) for k in range(lo, K + 1)]
            if K > lo:
                ops.propagate_chain(g, [(dhs[k + 1], dhs[k], dhs[k]) for k in range(K - 1, lo - 1, -1)], transpose=True, internal=True)
        else:
            dhs = [None] * (K + 1)
            dhs[K] = gk = ops.gemm([(dout, weights[K])], N, Fi, False, False, precision=precision)
            for k in range(K - 1, lo - 1, -1):
                dhk = ops.gemm([(dout, weights[k])], N, Fi, False, False, precision=precision)
                dhs[k] = gk = g.propagate(gk, transpose=True, add=dhk, internal=True)
    dx = g.from_internal(dhs[0]) if need_dx else dout.new_empty(0)
    return dx, db, dws, dhs, hs


@tag_conv_backward.register_fake
def _(dout, out, x, hops, edge_index, weights, relu, normalize, precision, ptr, need_dx, need_db, need_dw):
    return (torch.empty_like(x) if need_dx else x.new_empty(0), x.new_empty(dout.shape[1]) if need_db else x.new_empty(0),
            x.new_empty((len(weights),) + tuple(weights[0].shape)) if need_dw else x.new_empty(0))


def _tag_setup(ctx, inputs, output):
    x, edge_index, weights, bias, relu, normalize, precision, ptr = inputs
    out, hops = output
    ctx.meta = (relu, normalize, precision, ptr, bias is not None, len(weights))
    ctx.save_for_backward(out, x, hops, edge_index, *weights)
    ctx.set_materialize_grads(False)


def _tag_backward(ctx, dout, dhops):
    relu, normalize, precision, ptr, has_bias, nw = ctx.meta
    out, x, hops, edge_index, *weights = ctx.saved_tensors
    if dout is None:
        return (None,) * 8
    need_dx = ctx.needs_input_grad[0]
    nig_w = ctx.needs_input_grad[2]
    need_dw = any(nig_w) if isinstance(nig_w, (list, tuple)) else bool(nig_w)
    need_db = has_bias and ctx.needs_input_grad[3]
    dx, db, dws = torch.ops.dcb200.tag_conv_backward(dout, out, x, hops, edge_index, list(weights), relu, normalize, precision,
                                                     ptr, need_dx, need_db, need_dw)
    return (dx if need_dx else None, None, list(dws.unbind(0)) if need_dw else None, db if need_db else None, None, None, None,
            None)


tag_conv.register_autograd(_tag_backward, setup_context=_tag_setup)


# ----------------------------------------------------------------------------------- TAGConv with edge weights
@_lib.custom_op("dcb200::tag_conv_weighted", mutates_args=())
def tag_conv_weighted(x: Tensor, edge_index: Tensor, edge_weight: Tensor, weights: List[Tensor], bias: Optional[Tensor], relu: bool,
                      normalize: bool, precision: int, ptr: Optional[List[int]]) -> Tuple[Tensor, Tensor]:
    """``tag_conv`` with PyG's ``edge_weight`` [E] (edge_index order): the hops run on the weighted view of the "tag" structure
    (``ops.weighted_view``: gcn_norm(add_self_loops=False) of the weights, or the raw weights without ``normalize``)."""
    g = ops.weighted_view(_csr(edge_index, x.shape[0], "tag", ptr), edge_weight, normalize)
    return _tag_forward(g, x, weights, bias, relu, precision)


@tag_conv_weighted.register_fake
def _(x, edge_index, edge_weight, weights, bias, relu, normalize, precision, ptr):
    K = len(weights) - 1
    return x.new_empty((x.shape[0], weights[0].shape[0])), x.new_empty((x.shape[0], max(K, 1) * x.shape[1]))


@_lib.custom_op("dcb200::tag_conv_weighted_backward", mutates_args=())
def tag_conv_weighted_backward(dout: Tensor, out: Tensor, x: Tensor, hops: Tensor, edge_index: Tensor, edge_weight: Tensor,
                               weights: List[Tensor], relu: bool, normalize: bool, precision: int, ptr: Optional[List[int]],
                               need_dx: bool, need_db: bool, need_dw: bool, need_dew: bool) -> Tuple[Tensor, Tensor, Tensor, Tensor]:
    """-> (dx, dbias, dW stacked, dedge_weight [E]); empty tensors for gradients that are not needed.  dL/dnorm_e =
    sum_k <G_{k+1}[dst], H_k[src]> in one SDDMM launch over the saved hops and the transposed chain's totals, then the
    normalisation backward (dc_gcn_norm_weighted_backward)."""
    g = ops.weighted_view(_csr(edge_index, x.shape[0], "tag", ptr), edge_weight, normalize, transpose=True)
    dx, db, dws, dhs, hs = _tag_backward_impl(g, dout, out, x, hops, weights, relu, precision, need_dx, need_db, need_dw,
                                              need_chain=need_dew)
    K = len(weights) - 1
    if need_dew and K > 0:
        s, _ = ops.edge_sddmm(g, [(dhs[k + 1], hs[k]) for k in range(K)])
        dew = ops.gcn_norm_backward(g, s) if normalize else s
    elif need_dew:
        dew = torch.zeros_like(edge_weight)     # K = 0: the output does not depend on the edges
    else:
        dew = x.new_empty(0)
    return dx, db, dws, dew


@tag_conv_weighted_backward.register_fake
def _(dout, out, x, hops, edge_index, edge_weight, weights, relu, normalize, precision, ptr, need_dx, need_db, need_dw, need_dew):
    return (torch.empty_like(x) if need_dx else x.new_empty(0), x.new_empty(dout.shape[1]) if need_db else x.new_empty(0),
            x.new_empty((len(weights),) + tuple(weights[0].shape)) if need_dw else x.new_empty(0),
            torch.empty_like(edge_weight) if need_dew else x.new_empty(0))


def _tag_w_setup(ctx, inputs, output):
    x, edge_index, edge_weight, weights, bias, relu, normalize, precision, ptr = inputs
    out, hops = output
    ctx.meta = (relu, normalize, precision, ptr, bias is not None, len(weights))
    ctx.save_for_backward(out, x, hops, edge_index, edge_weight, *weights)
    ctx.set_materialize_grads(False)


def _tag_w_backward(ctx, dout, dhops):
    relu, normalize, precision, ptr, has_bias, nw = ctx.meta
    out, x, hops, edge_index, edge_weight, *weights = ctx.saved_tensors
    if dout is None:
        return (None,) * 9
    need_dx, need_dew = ctx.needs_input_grad[0], ctx.needs_input_grad[2]
    nig_w = ctx.needs_input_grad[3]
    need_dw = any(nig_w) if isinstance(nig_w, (list, tuple)) else bool(nig_w)
    need_db = has_bias and ctx.needs_input_grad[4]
    dx, db, dws, dew = torch.ops.dcb200.tag_conv_weighted_backward(dout, out, x, hops, edge_index, edge_weight, list(weights), relu,
                                                                   normalize, precision, ptr, need_dx, need_db, need_dw, need_dew)
    return (dx if need_dx else None, None, dew if need_dew else None, list(dws.unbind(0)) if need_dw else None,
            db if need_db else None, None, None, None, None)


tag_conv_weighted.register_autograd(_tag_w_backward, setup_context=_tag_w_setup)


# ----------------------------------------------------------------------------------- GCNConv
@_lib.custom_op("dcb200::gcn_conv", mutates_args=())
def gcn_conv(x: Tensor, edge_index: Tensor, weight: Tensor, bias: Optional[Tensor], relu: bool, precision: int,
             ptr: Optional[List[int]]) -> Tensor:
    g = _csr(edge_index, x.shape[0], "gcn", ptr)
    xw = ops.gemm([(x.contiguous(), weight)], x.shape[0], weight.shape[0], False, True, precision=precision)
    return g.propagate(xw, bias=bias, relu=relu)


@gcn_conv.register_fake
def _(x, edge_index, weight, bias, relu, precision, ptr):
    return x.new_empty((x.shape[0], weight.shape[0]))


@_lib.custom_op("dcb200::gcn_conv_backward", mutates_args=())
def gcn_conv_backward(dout: Tensor, out: Tensor, x: Tensor, edge_index: Tensor, weight: Tensor, relu: bool, precision: int,
                      ptr: Optional[List[int]], need_dx: bool, need_db: bool) -> Tuple[Tensor, Tensor, Tensor]:
    g = _csr(edge_index, x.shape[0], "gcn", ptr)
    dout, db = ops.relu_bwd_db(out, dout.contiguous(), relu, need_db)
    N, Fo = dout.shape
    Fi = x.shape[1]
    db = db if need_db else dout.new_empty(0)
    dxw = g.propagate(dout, transpose=True)
    dx = ops.gemm([(dxw, weight)], N, Fi, False, False, precision=precision) if need_dx else dout.new_empty(0)
    dw = ops.gemm([(dxw, x.contiguous())], Fo, Fi, True, False, precision=precision)
    return dx, dw, db


@gcn_conv_backward.register_fake
def _(dout, out, x, edge_index, weight, relu, precision, ptr, need_dx, need_db):
    return (torch.empty_like(x) if need_dx else x.new_empty(0), torch.empty_like(weight),
            x.new_empty(dout.shape[1]) if need_db else x.new_empty(0))


def _gcn_setup(ctx, inputs, output):
    x, edge_index, weight, bias, relu, precision, ptr = inputs
    ctx.meta = (relu, precision, ptr, bias is not None)
    ctx.save_for_backward(output, x, edge_index, weight)


def _gcn_backward(ctx, dout):
    relu, precision, ptr, has_bias = ctx.meta
    out, x, edge_index, weight = ctx.saved_tensors
    need_dx, need_db = ctx.needs_input_grad[0], has_bias and ctx.needs_input_grad[3]
    dx, dw, db = torch.ops.dcb200.gcn_conv_backward(dout, out, x, edge_index, weight, relu, precision, ptr, need_dx, need_db)
    return (dx if need_dx else None, None, dw, db if need_db else None, None, None, None)


gcn_conv.register_autograd(_gcn_backward, setup_context=_gcn_setup)


# ----------------------------------------------------------------------------------- GCNConv with edge weights
@_lib.custom_op("dcb200::gcn_conv_weighted", mutates_args=())
def gcn_conv_weighted(x: Tensor, edge_index: Tensor, edge_weight: Tensor, weight: Tensor, bias: Optional[Tensor], relu: bool,
                      fill_value: float, precision: int, ptr: Optional[List[int]]) -> Tuple[Tensor, Tensor]:
    """``gcn_conv`` with PyG's ``edge_weight`` [E] (edge_index order) and ``add_remaining_self_loops(fill_value)`` (2 for
    ``improved``): -> (out, xw = x W^T, kept for the backward)."""
    g = ops.weighted_view(_csr(edge_index, x.shape[0], "gcn", ptr), edge_weight, True, fill_value)
    xw = ops.gemm([(x.contiguous(), weight)], x.shape[0], weight.shape[0], False, True, precision=precision)
    return g.propagate(xw, bias=bias, relu=relu), xw


@gcn_conv_weighted.register_fake
def _(x, edge_index, edge_weight, weight, bias, relu, fill_value, precision, ptr):
    return x.new_empty((x.shape[0], weight.shape[0])), x.new_empty((x.shape[0], weight.shape[0]))


@_lib.custom_op("dcb200::gcn_conv_weighted_backward", mutates_args=())
def gcn_conv_weighted_backward(dout: Tensor, out: Tensor, x: Tensor, xw: Tensor, edge_index: Tensor, edge_weight: Tensor,
                               weight: Tensor, relu: bool, fill_value: float, precision: int, ptr: Optional[List[int]],
                               need_dx: bool, need_db: bool, need_dew: bool) -> Tuple[Tensor, Tensor, Tensor, Tensor]:
    """-> (dx, dW, dbias, dedge_weight [E]); dL/dnorm_e = <dOut[dst], xw[src]> and the loop's <dOut[i], xw[i]> in one SDDMM
    launch, then the normalisation backward."""
    g = ops.weighted_view(_csr(edge_index, x.shape[0], "gcn", ptr), edge_weight, True, fill_value, transpose=True)
    dout, db = ops.relu_bwd_db(out, dout.contiguous(), relu, need_db)
    N, Fo = dout.shape
    Fi = x.shape[1]
    db = db if need_db else dout.new_empty(0)
    dxw = g.propagate(dout, transpose=True)
    dx = ops.gemm([(dxw, weight)], N, Fi, False, False, precision=precision) if need_dx else dout.new_empty(0)
    dw = ops.gemm([(dxw, x.contiguous())], Fo, Fi, True, False, precision=precision)
    if need_dew:
        s, s_self = ops.edge_sddmm(g, [(g.to_internal(dout), g.to_internal(xw.contiguous()))], self_term=True)
        dew = ops.gcn_norm_backward(g, s, s_self)
    else:
        dew = dout.new_empty(0)
    return dx, dw, db, dew


@gcn_conv_weighted_backward.register_fake
def _(dout, out, x, xw, edge_index, edge_weight, weight, relu, fill_value, precision, ptr, need_dx, need_db, need_dew):
    return (torch.empty_like(x) if need_dx else x.new_empty(0), torch.empty_like(weight),
            x.new_empty(dout.shape[1]) if need_db else x.new_empty(0), torch.empty_like(edge_weight) if need_dew else x.new_empty(0))


def _gcn_w_setup(ctx, inputs, output):
    x, edge_index, edge_weight, weight, bias, relu, fill_value, precision, ptr = inputs
    out, xw = output
    ctx.meta = (relu, fill_value, precision, ptr, bias is not None)
    ctx.save_for_backward(out, x, xw, edge_index, edge_weight, weight)
    ctx.set_materialize_grads(False)


def _gcn_w_backward(ctx, dout, dxw):
    relu, fill_value, precision, ptr, has_bias = ctx.meta
    out, x, xw, edge_index, edge_weight, weight = ctx.saved_tensors
    if dout is None:
        return (None,) * 9
    need_dx, need_dew, need_db = ctx.needs_input_grad[0], ctx.needs_input_grad[2], has_bias and ctx.needs_input_grad[4]
    dx, dw, db, dew = torch.ops.dcb200.gcn_conv_weighted_backward(dout, out, x, xw, edge_index, edge_weight, weight, relu, fill_value,
                                                                  precision, ptr, need_dx, need_db, need_dew)
    return (dx if need_dx else None, None, dew if need_dew else None, dw, db if need_db else None, None, None, None, None)


gcn_conv_weighted.register_autograd(_gcn_w_backward, setup_context=_gcn_w_setup)


# ----------------------------------------------------------------------------------- GATConv (heads = 1)
@_lib.custom_op("dcb200::gat_conv", mutates_args=())
def gat_conv(x: Tensor, edge_index: Tensor, weight: Tensor, att_src: Tensor, att_dst: Tensor, bias: Optional[Tensor],
             negative_slope: float, relu: bool, precision: int,
             ptr: Optional[List[int]]) -> Tuple[Tensor, Tensor, Tensor, Tensor, Tensor, Tensor]:
    """PyG 2.5.x GATConv (heads=1, add_self_loops; models/model.py:39,71,77): xs = x W^T; a_s = xs.att_src, a_d = xs.att_dst;
    per-receiver softmax over leaky_relu(a_s[j] + a_d[i]) incl. the appended self loop; out = sum alpha xs[j] + b.
    -> (out, xs, a_src, a_dst, alpha_edge, alpha_self); all but ``out`` are kept for the backward."""
    g = _csr(edge_index, x.shape[0], "gat", ptr)
    x = x.contiguous()
    N, C_ = x.shape[0], weight.shape[0]
    xs = ops.gemm([(x, weight)], N, C_, False, True, precision=precision)
    a_src, a_dst = ops.gat_scores(xs, att_src.reshape(-1), att_dst.reshape(-1), 1, C_)
    alpha_e, alpha_s = ops.gat_softmax(g, a_src, a_dst, negative_slope)
    out = ops.spmm(g.rowptr, g.nbr, xs, edge_w=alpha_e, edge_w_index=g.eid, self_w=alpha_s, self_loop=True, bias=bias, relu=relu)
    return out, xs, a_src, a_dst, alpha_e, alpha_s


@gat_conv.register_fake
def _(x, edge_index, weight, att_src, att_dst, bias, negative_slope, relu, precision, ptr):
    N, C_ = x.shape[0], weight.shape[0]
    return (x.new_empty((N, C_)), x.new_empty((N, C_)), x.new_empty((N, 1)), x.new_empty((N, 1)),
            x.new_empty(max(edge_index.shape[1], 1)), x.new_empty(N))


@_lib.custom_op("dcb200::gat_conv_backward", mutates_args=())
def gat_conv_backward(dout: Tensor, out: Tensor, x: Tensor, edge_index: Tensor, weight: Tensor, att_src: Tensor, att_dst: Tensor,
                      xs: Tensor, a_src: Tensor, a_dst: Tensor, alpha_e: Tensor, alpha_s: Tensor, negative_slope: float, relu: bool,
                      precision: int, ptr: Optional[List[int]], need_dx: bool,
                      need_db: bool) -> Tuple[Tensor, Tensor, Tensor, Tensor, Tensor]:
    """-> (dx, dW, datt_src, datt_dst, dbias); empty tensors for gradients that are not needed."""
    g = _csr(edge_index, x.shape[0], "gat", ptr)
    dout, db = ops.relu_bwd_db(out, dout.contiguous(), relu, need_db)
    N, C_ = dout.shape
    Fi = x.shape[1]
    x = x.contiguous()
    db = db if need_db else dout.new_empty(0)
    rpt, nbt, eidt = g.t
    # through the aggregation: dxs[j] = sum_{e: src=j} alpha_e dout[dst_e] + alpha_self[j] dout[j]
    dz_e, dz_s, da_dst = ops.gat_bwd_edge(g, a_src, a_dst, negative_slope, alpha_e, alpha_s, xs, dout)
    da_src = ops.segment_sum(rpt, eidt, dz_e, dz_s, N)
    # through the scores: dxs += da_src (x) att_src + da_dst (x) att_dst  == [da_src da_dst] @ [att_src; att_dst]
    da = torch.stack([da_src, da_dst], 1).contiguous()                       # [N, 2]
    att = torch.cat([att_src.reshape(1, -1), att_dst.reshape(1, -1)], 0).contiguous()  # [2, C]
    dxs0 = ops.gemm([(da, att)], N, C_, False, False, precision=ops.GEMM_FP32)
    dxs = ops.spmm(rpt, nbt, dout, edge_w=alpha_e, edge_w_index=eidt, self_w=alpha_s, self_loop=True, add=dxs0)
    datt = ops.gemm([(da, xs)], 2, C_, True, False, precision=ops.GEMM_FP32)  # [2, C] = da^T xs
    dx = ops.gemm([(dxs, weight)], N, Fi, False, False, precision=precision) if need_dx else dout.new_empty(0)
    dw = ops.gemm([(dxs, x)], C_, Fi, True, False, precision=precision)
    return dx, dw, datt[0].reshape(att_src.shape).clone(), datt[1].reshape(att_dst.shape).clone(), db


@gat_conv_backward.register_fake
def _(dout, out, x, edge_index, weight, att_src, att_dst, xs, a_src, a_dst, alpha_e, alpha_s, negative_slope, relu, precision, ptr,
      need_dx, need_db):
    return (torch.empty_like(x) if need_dx else x.new_empty(0), torch.empty_like(weight), torch.empty_like(att_src),
            torch.empty_like(att_dst), x.new_empty(dout.shape[1]) if need_db else x.new_empty(0))


def _gat_setup(ctx, inputs, output):
    x, edge_index, weight, att_src, att_dst, bias, slope, relu, precision, ptr = inputs
    out, xs, a_src, a_dst, alpha_e, alpha_s = output
    ctx.meta = (slope, relu, precision, ptr, bias is not None)
    ctx.save_for_backward(out, x, edge_index, weight, att_src, att_dst, xs, a_src, a_dst, alpha_e, alpha_s)
    ctx.set_materialize_grads(False)


def _gat_backward(ctx, dout, *_unused):
    slope, relu, precision, ptr, has_bias = ctx.meta
    out, x, edge_index, weight, att_src, att_dst, xs, a_src, a_dst, alpha_e, alpha_s = ctx.saved_tensors
    if dout is None:
        return (None,) * 10
    need_dx, need_db = ctx.needs_input_grad[0], has_bias and ctx.needs_input_grad[5]
    dx, dw, das, dad, db = torch.ops.dcb200.gat_conv_backward(dout, out, x, edge_index, weight, att_src, att_dst, xs, a_src, a_dst,
                                                              alpha_e, alpha_s, slope, relu, precision, ptr, need_dx, need_db)
    return (dx if need_dx else None, None, dw, das, dad, db if need_db else None, None, None, None, None)


gat_conv.register_autograd(_gat_backward, setup_context=_gat_setup)


# ----------------------------------------------------------------------------------- GATConv (any heads)
@_lib.custom_op("dcb200::gat_conv_heads", mutates_args=())
def gat_conv_heads(x: Tensor, edge_index: Tensor, weight: Tensor, att_src: Tensor, att_dst: Tensor, bias: Optional[Tensor],
                   negative_slope: float, heads: int, concat: bool, relu: bool, precision: int,
                   ptr: Optional[List[int]]) -> Tuple[Tensor, Tensor, Tensor, Tensor, Tensor, Tensor]:
    """PyG 2.5.x GATConv(heads=H, concat=...): xs = x W^T viewed as [N, H, C]; per head a_s, a_d, the per-receiver softmax incl.
    the appended self loop and the weighted sum; out = [N, H*C] (concat) or the mean over heads [N, C], + bias.  Softmax and
    aggregation are one launch (dc_gat_aggregate).  -> (out, xs, a_src [N, H], a_dst [N, H], alpha_edge [max(E,1), H],
    alpha_self [N, H]); all but ``out`` are kept for the backward."""
    g = _csr(edge_index, x.shape[0], "gat", ptr)
    x = x.contiguous()
    N, HC = x.shape[0], weight.shape[0]
    C_ = HC // heads
    xs = ops.gemm([(x, weight)], N, HC, False, True, precision=precision)
    a_src, a_dst = ops.gat_scores(xs, att_src.reshape(-1), att_dst.reshape(-1), heads, C_)
    out, alpha_e, alpha_s = ops.gat_aggregate(g, xs, a_src, a_dst, negative_slope, heads, C_, concat, bias=bias, relu=relu)
    return out, xs, a_src, a_dst, alpha_e, alpha_s


@gat_conv_heads.register_fake
def _(x, edge_index, weight, att_src, att_dst, bias, negative_slope, heads, concat, relu, precision, ptr):
    N, HC = x.shape[0], weight.shape[0]
    return (x.new_empty((N, HC if concat else HC // heads)), x.new_empty((N, HC)), x.new_empty((N, heads)), x.new_empty((N, heads)),
            x.new_empty((max(edge_index.shape[1], 1), heads)), x.new_empty((N, heads)))


@_lib.custom_op("dcb200::gat_conv_heads_backward", mutates_args=())
def gat_conv_heads_backward(dout: Tensor, out: Tensor, x: Tensor, edge_index: Tensor, weight: Tensor, att_src: Tensor,
                            att_dst: Tensor, xs: Tensor, a_src: Tensor, a_dst: Tensor, alpha_e: Tensor, alpha_s: Tensor,
                            negative_slope: float, heads: int, concat: bool, relu: bool, precision: int, ptr: Optional[List[int]],
                            need_dx: bool, need_db: bool, dalpha_e: Optional[Tensor] = None,
                            dalpha_s: Optional[Tensor] = None) -> Tuple[Tensor, Tensor, Tensor, Tensor, Tensor]:
    """-> (dx, dW, datt_src, datt_dst, dbias); empty tensors for gradients that are not needed.  dz and da_dst by receiver
    (dc_gat_bwd_edge_heads), then dxs and da_src in one pass by source (dc_gat_scatter_heads), datt by a column reduction.
    ``dalpha_e`` [max(E,1), H] / ``dalpha_s`` [N, H]: the gradient of the loss wrt the attention coefficients themselves, added
    to the one through the aggregation by the receiver pass (dc_gat_bwd_edge_heads_ext); the other passes are unchanged."""
    g = _csr(edge_index, x.shape[0], "gat", ptr)
    dout, db = ops.relu_bwd_db(out, dout.contiguous(), relu, need_db)
    N, Fi = x.shape
    HC = weight.shape[0]
    C_ = HC // heads
    x = x.contiguous()
    db = db if need_db else dout.new_empty(0)
    dz_e, dz_s, da_dst = ops.gat_bwd_edge_heads(g, a_src, a_dst, negative_slope, alpha_e, alpha_s, xs, dout, heads, C_, concat,
                                                dalpha_e, dalpha_s)
    dxs, da_src = ops.gat_scatter_heads(g, alpha_e, alpha_s, dz_e, dz_s, da_dst, att_src, att_dst, dout, heads, C_, concat)
    datt_s, datt_d = ops.gat_att_grad(xs, da_src, da_dst, heads, C_)
    dx = ops.gemm([(dxs, weight)], N, Fi, False, False, precision=precision) if need_dx else dout.new_empty(0)
    dw = ops.gemm([(dxs, x)], HC, Fi, True, False, precision=precision)
    return dx, dw, datt_s.reshape(att_src.shape), datt_d.reshape(att_dst.shape), db


@gat_conv_heads_backward.register_fake
def _(dout, out, x, edge_index, weight, att_src, att_dst, xs, a_src, a_dst, alpha_e, alpha_s, negative_slope, heads, concat, relu,
      precision, ptr, need_dx, need_db, dalpha_e=None, dalpha_s=None):
    return (torch.empty_like(x) if need_dx else x.new_empty(0), torch.empty_like(weight), torch.empty_like(att_src),
            torch.empty_like(att_dst), x.new_empty(dout.shape[1]) if need_db else x.new_empty(0))


def _gat_heads_setup(ctx, inputs, output):
    x, edge_index, weight, att_src, att_dst, bias, slope, heads, concat, relu, precision, ptr = inputs
    out, xs, a_src, a_dst, alpha_e, alpha_s = output
    ctx.meta = (slope, heads, concat, relu, precision, ptr, bias is not None)
    ctx.save_for_backward(out, x, edge_index, weight, att_src, att_dst, xs, a_src, a_dst, alpha_e, alpha_s)
    ctx.set_materialize_grads(False)


def _gat_heads_backward(ctx, dout, _dxs, _da_src, _da_dst, dalpha_e, dalpha_s):
    slope, heads, concat, relu, precision, ptr, has_bias = ctx.meta
    out, x, edge_index, weight, att_src, att_dst, xs, a_src, a_dst, alpha_e, alpha_s = ctx.saved_tensors
    if dout is None and dalpha_e is None and dalpha_s is None:
        return (None,) * 12
    need_dx, need_db = ctx.needs_input_grad[0], has_bias and ctx.needs_input_grad[5] and dout is not None
    if dout is None:
        dout = torch.zeros_like(out)      # a loss on alpha alone: the kernels read zeros (the bias gets no gradient)
    dalpha_e = dalpha_e.contiguous() if dalpha_e is not None else None
    dalpha_s = dalpha_s.contiguous() if dalpha_s is not None else None
    dx, dw, das, dad, db = torch.ops.dcb200.gat_conv_heads_backward(dout, out, x, edge_index, weight, att_src, att_dst, xs, a_src,
                                                                    a_dst, alpha_e, alpha_s, slope, heads, concat, relu, precision,
                                                                    ptr, need_dx, need_db, dalpha_e, dalpha_s)
    return (dx if need_dx else None, None, dw, das, dad, db if need_db else None, None, None, None, None, None, None)


gat_conv_heads.register_autograd(_gat_heads_backward, setup_context=_gat_heads_setup)


# ----------------------------------------------------------------------------------- MPNN layer (A9 extension)
@_lib.custom_op("dcb200::mpnn_layer", mutates_args=())
def mpnn_layer(x: Tensor, edge_index: Tensor, We1: Tensor, be1: Tensor, We2: Tensor, be2: Tensor, Wn1: Tensor, bn1: Tensor,
               Wn2: Tensor, bn2: Tensor, residual: bool, precision: int,
               ptr: Optional[List[int]]) -> Tuple[Tensor, Tensor, Tensor, Tensor, Tensor, Tensor]:
    """Edge-MLP / scatter-sum / node-MLP residual layer (north_star wording; no reference symbol):
        m_e = W_e2 relu(W_e1 [x_i || x_j] + b_e1) + b_e2,  a_i = sum_{e: dst = i} m_e,
        x'_i = x_i + W_n2 relu(W_n1 [x_i || a_i] + b_n1) + b_n2.
    The first edge Linear is split into two NODE-level GEMMs (u = x W_e1[:, :F]^T + b, v = x W_e1[:, F:]^T) and, because the
    aggregation is a sum, the second edge Linear moves outside it: a = (sum_e relu(u_i + v_j)) W_e2^T + deg * b_e2.
    Per-edge work is one fused gather (dc_edge_relu); edge features never exist in HBM.
    -> (out, u, v, s, a, h1); all but ``out`` are kept for the backward."""
    g = _csr(edge_index, x.shape[0], "plain", ptr)
    x = x.contiguous()
    N, Fi = x.shape
    Fo = We2.shape[0]
    u = ops.gemm([(x, We1[:, :Fi])], N, Fo, False, True, bias=be1, precision=precision)
    v = ops.gemm([(x, We1[:, Fi:])], N, Fo, False, True, precision=precision)
    s = ops.edge_relu(g.rowptr, g.nbr, u, v, mode=0)
    deg = (g.rowptr[1:] - g.rowptr[:-1]).to(x.dtype).unsqueeze(1)
    a = ops.gemm([(s, We2)], N, Fo, False, True, precision=precision)
    a.addcmul_(deg, be2.unsqueeze(0))
    h1 = ops.gemm([(x, Wn1[:, :Fi]), (a, Wn1[:, Fi:])], N, Fo, False, True, bias=bn1, relu=True, precision=precision)
    if residual:
        out = x.clone()
        ops.gemm([(h1, Wn2)], N, Fo, False, True, bias=bn2, out=out, accumulate=True, precision=precision)
    else:
        out = ops.gemm([(h1, Wn2)], N, Fo, False, True, bias=bn2, precision=precision)
    return out, u, v, s, a, h1


@mpnn_layer.register_fake
def _(x, edge_index, We1, be1, We2, be2, Wn1, bn1, Wn2, bn2, residual, precision, ptr):
    N, Fo = x.shape[0], We2.shape[0]
    return tuple(x.new_empty((N, Fo)) for _ in range(6))


@_lib.custom_op("dcb200::mpnn_layer_backward", mutates_args=())
def mpnn_layer_backward(dout: Tensor, x: Tensor, edge_index: Tensor, u: Tensor, v: Tensor, s: Tensor, a: Tensor, h1: Tensor,
                        We1: Tensor, We2: Tensor, Wn1: Tensor, Wn2: Tensor, residual: bool, precision: int,
                        ptr: Optional[List[int]]) -> Tuple[Tensor, Tensor, Tensor, Tensor, Tensor, Tensor, Tensor, Tensor, Tensor]:
    """-> (dx, dWe1, dbe1, dWe2, dbe2, dWn1, dbn1, dWn2, dbn2)."""
    g = _csr(edge_index, x.shape[0], "plain", ptr)
    P = precision
    dout, x = dout.contiguous(), x.contiguous()
    N, Fi = x.shape
    Fo = We2.shape[0]
    G = ops.gemm
    deg = (g.rowptr[1:] - g.rowptr[:-1]).to(x.dtype).unsqueeze(1)
    dh1 = ops.relu_bwd(h1, G([(dout, Wn2)], N, Fo, False, False, precision=P))
    dWn2, dbn2 = G([(dout, h1)], Fo, Fo, True, False, precision=P), ops.colsum(dout)
    dWn1 = torch.empty_like(Wn1)
    G([(dh1, x)], Fo, Fi, True, False, out=dWn1[:, :Fi], precision=P)
    G([(dh1, a)], Fo, Fo, True, False, out=dWn1[:, Fi:], precision=P)
    dbn1 = ops.colsum(dh1)
    dx = dout.clone() if residual else torch.zeros_like(x)
    G([(dh1, Wn1[:, :Fi])], N, Fi, False, False, out=dx, accumulate=True, precision=P)
    da = G([(dh1, Wn1[:, Fi:])], N, Fo, False, False, precision=P)
    dWe2 = G([(da, s)], Fo, Fo, True, False, precision=P)
    dbe2 = ops.colsum(da * deg)
    ds = G([(da, We2)], N, Fo, False, False, precision=P)
    du = ops.edge_relu(g.rowptr, g.nbr, u, v, ds, mode=1)
    rpt, nbt, _ = g.t
    dv = ops.edge_relu(rpt, nbt, v, u, ds, mode=2)
    dWe1 = torch.empty_like(We1)
    G([(du, x)], Fo, Fi, True, False, out=dWe1[:, :Fi], precision=P)
    G([(dv, x)], Fo, Fi, True, False, out=dWe1[:, Fi:], precision=P)
    dbe1 = ops.colsum(du)
    G([(du, We1[:, :Fi])], N, Fi, False, False, out=dx, accumulate=True, precision=P)
    G([(dv, We1[:, Fi:])], N, Fi, False, False, out=dx, accumulate=True, precision=P)
    return dx, dWe1, dbe1, dWe2, dbe2, dWn1, dbn1, dWn2, dbn2


@mpnn_layer_backward.register_fake
def _(dout, x, edge_index, u, v, s, a, h1, We1, We2, Wn1, Wn2, residual, precision, ptr):
    Fo = We2.shape[0]
    return (torch.empty_like(x), torch.empty_like(We1), x.new_empty(Fo), torch.empty_like(We2), x.new_empty(Fo),
            torch.empty_like(Wn1), x.new_empty(Fo), torch.empty_like(Wn2), x.new_empty(Fo))


def _mpnn_setup(ctx, inputs, output):
    x, edge_index, We1, be1, We2, be2, Wn1, bn1, Wn2, bn2, residual, precision, ptr = inputs
    out, u, v, s, a, h1 = output
    ctx.meta = (residual, precision, ptr)
    ctx.save_for_backward(x, edge_index, u, v, s, a, h1, We1, We2, Wn1, Wn2)
    ctx.set_materialize_grads(False)


def _mpnn_backward(ctx, dout, *_unused):
    residual, precision, ptr = ctx.meta
    x, edge_index, u, v, s, a, h1, We1, We2, Wn1, Wn2 = ctx.saved_tensors
    if dout is None:
        return (None,) * 13
    dx, dWe1, dbe1, dWe2, dbe2, dWn1, dbn1, dWn2, dbn2 = torch.ops.dcb200.mpnn_layer_backward(
        dout, x, edge_index, u, v, s, a, h1, We1, We2, Wn1, Wn2, residual, precision, ptr)
    return (dx if ctx.needs_input_grad[0] else None, None, dWe1, dbe1, dWe2, dbe2, dWn1, dbn1, dWn2, dbn2, None, None, None)


mpnn_layer.register_autograd(_mpnn_backward, setup_context=_mpnn_setup)


# ----------------------------------------------------------------------------------- edge builders (edge_index level)
def _dynamic_edges(pos):
    ctx = torch.library.get_ctx()
    n_edges, n_order = ctx.new_dynamic_size(), ctx.new_dynamic_size()     # both data dependent (E; 0 or N)
    return (torch.empty((2, n_edges), dtype=torch.int64, device=pos.device), torch.empty(n_order, dtype=torch.int32, device=pos.device))


@_lib.custom_op("dcb200::knn_graph", mutates_args=())
def knn_graph(pos: Tensor, k: int, batch: Optional[Tensor], loop: bool, ptr: Optional[Tensor]) -> Tuple[Tensor, Tensor]:
    """torch_cluster.knn_graph(pos, k, batch, loop, flow='source_to_target') (utils/pointcloud_utils.py:12) -> (edge_index int64
    [2, E], cell order int32 [N] of a single large cloud for ops.register_order_hint, else empty).  E is data dependent."""
    tab = ops.knn_table(pos, k, batch=batch, ptr=ptr, loop=loop)
    order = getattr(tab, "_cell_order", None)
    return ops.table_to_edge_index(tab), (order if order is not None else torch.empty(0, dtype=torch.int32, device=pos.device))


@knn_graph.register_fake
def _(pos, k, batch, loop, ptr):
    return _dynamic_edges(pos)


@_lib.custom_op("dcb200::radius_graph", mutates_args=())
def radius_graph(pos: Tensor, r: float, batch: Optional[Tensor], loop: bool, max_num_neighbors: int,
                 ptr: Optional[Tensor]) -> Tuple[Tensor, Tensor]:
    """torch_cluster.radius_graph(pos, r, batch, loop, max_num_neighbors) (utils/pointcloud_utils.py:10) -> (edge_index, cell order)."""
    tab, _ = ops.radius_table(pos, r, batch=batch, ptr=ptr, loop=loop, max_num_neighbors=max_num_neighbors)
    order = getattr(tab, "_cell_order", None)
    return ops.table_to_edge_index(tab), (order if order is not None else torch.empty(0, dtype=torch.int32, device=pos.device))


@radius_graph.register_fake
def _(pos, r, batch, loop, max_num_neighbors, ptr):
    return _dynamic_edges(pos)
