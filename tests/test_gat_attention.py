"""CPU tests of GATConv's ``return_attention_weights``: the reference (tests/gat_attention_reference.py) against a dense fp64
formulation, the order of ``edge_index_sl``, normalisation of alpha, an fp64 gradcheck of a loss on alpha, and the return forms
and signature of the drop-in layer."""
import inspect
import os
import re

import pytest
import torch

from helpers import assert_close
from gat_attention_reference import GATConvAttention
from oracle import convs

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _g(seed=0, n=60, e=400, f=21):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(n, f, generator=g), torch.randint(0, n, (2, e), generator=g)


def _layer(heads, concat, seed=0, C=8, dtype=torch.float32):
    torch.manual_seed(seed)
    layer = GATConvAttention(21, C, heads=heads, concat=concat)
    with torch.no_grad():
        layer.bias.uniform_(-0.5, 0.5)
    return layer.to(dtype)


@pytest.mark.parametrize("heads,concat", [(1, True), (3, True), (2, False)])
def test_reference_vs_dense_fp64(heads, concat):
    """Per head the dense masked softmax P [receiver, sender] (self loop included): alpha[r] = P[col_r, row_r], out = P xs."""
    x, ei = _g(1)
    ei = torch.unique(ei, dim=1)       # the dense form cannot express duplicates; input self loops stay (they are replaced)
    layer = _layer(heads, concat)
    out, (ei_sl, alpha) = layer(x, ei, return_attention_weights=True)
    n, C = x.shape[0], layer.out_channels
    xs = (x.double() @ layer.lin.weight.double().t()).view(n, heads, C)
    mask = torch.eye(n, dtype=torch.bool)
    mask[ei[1], ei[0]] = True
    outs, alphas = [], []
    for h in range(heads):
        a_s, a_d = xs[:, h] @ layer.att_src[0, h].double(), xs[:, h] @ layer.att_dst[0, h].double()
        e = torch.nn.functional.leaky_relu(a_d[:, None] + a_s[None, :], layer.negative_slope).masked_fill(~mask, float("-inf"))
        P = torch.softmax(e, dim=1)
        outs.append(P @ xs[:, h])
        alphas.append(P[ei_sl[1], ei_sl[0]])
    dense = (torch.cat(outs, 1) if concat else torch.stack(outs, 0).mean(0)) + layer.bias.double()
    assert alpha.shape == (ei_sl.shape[1], heads) and alpha.dtype == torch.float32
    assert_close(out, dense.float(), what=f"out H={heads} concat={concat}")
    assert_close(alpha, torch.stack(alphas, 1).float(), what=f"alpha H={heads} concat={concat}")


def test_alpha_of_each_receiver_sums_to_one():
    x, ei = _g(2, n=80, e=500)
    ei = torch.cat([ei[:, :, None].expand(2, 500, 2).reshape(2, -1), torch.arange(5).repeat(2, 1)], 1)  # duplicates, loops
    ei = ei[:, ei.max(0).values < 70]                          # nodes 70..79 only have their appended loop
    layer = _layer(4, True)
    _, (ei_sl, alpha) = layer(x, ei, return_attention_weights=True)
    sums = convs._scatter_sum(alpha.double(), ei_sl[1], x.shape[0])
    assert_close(sums, torch.ones_like(sums), what="sum of alpha per receiver")
    assert torch.equal(alpha[-10:], torch.ones(10, 4))        # isolated nodes attend to themselves only


def test_edge_index_sl_order_with_duplicates_and_self_loops():
    ei = torch.tensor([[0, 2, 1, 2, 3, 0, 3, 1],
                       [1, 2, 0, 2, 0, 1, 3, 0]])
    x = torch.randn(5, 21, generator=torch.Generator().manual_seed(0))
    _, (ei_sl, alpha) = _layer(2, False)(x, ei, return_attention_weights=True)
    expect = torch.tensor([[0, 1, 3, 0, 1, 0, 1, 2, 3, 4],
                           [1, 0, 0, 1, 0, 0, 1, 2, 3, 4]])
    assert ei_sl.dtype == torch.int64 and torch.equal(ei_sl, expect)
    assert alpha.shape == (10, 2)
    assert torch.equal(alpha[0], alpha[3]) and torch.equal(alpha[1], alpha[4])   # duplicate edges share their coefficient


def test_gradcheck_of_a_loss_on_alpha_fp64():
    x, ei = _g(3, n=12, e=40)
    layer = _layer(2, True, C=3, dtype=torch.float64)
    names = ["lin.weight", "att_src", "att_dst", "bias"]
    params = [dict(layer.named_parameters())[k].detach().clone().requires_grad_(True) for k in names]
    x = x.double().requires_grad_(True)

    def f(x_, *ps):
        out, (_, alpha) = torch.func.functional_call(layer, dict(zip(names, ps)), (x_, ei), {"return_attention_weights": True})
        return out, alpha

    assert torch.autograd.gradcheck(lambda *a: f(*a)[1], (x, *params[:3], params[3].detach()))
    assert torch.autograd.gradcheck(f, (x, *params))


def test_reference_return_forms():
    x, ei = _g(4)
    layer = _layer(2, True)
    out = layer(x, ei)
    assert isinstance(out, torch.Tensor)
    for flag in (True, False):
        res = layer(x, ei, return_attention_weights=flag)
        assert isinstance(res, tuple) and len(res) == 2 and torch.equal(res[0], out)


def test_layer_signature_and_rejected_flags():
    import deformcontact_b200 as dc
    sig = inspect.signature(dc.GATConv.forward)
    assert list(sig.parameters)[:5] == ["self", "x", "edge_index", "relu", "ptr"]
    p = sig.parameters["return_attention_weights"]
    assert p.kind is inspect.Parameter.KEYWORD_ONLY and p.default is None
    layer = dc.GATConv(21, 8, heads=2)
    ours_ref = GATConvAttention(21, 8, heads=2)
    ours_ref.load_state_dict(layer.state_dict())              # the keys are PyG's both ways
    layer.load_state_dict(ours_ref.state_dict())
    x, ei = _g(5)
    for bad in (1, 0, "yes", torch.tensor(True)):
        with pytest.raises(TypeError):
            layer(x, ei, return_attention_weights=bad)
    with pytest.raises(TypeError):
        layer(x, ei, False, None, True)                         # keyword only


def test_extended_entry_point_is_declared_and_bound():
    from deformcontact_b200 import _abi
    import deformcontact_b200  # noqa: F401  (registers the ops)
    hdr = open(os.path.join(ROOT, "include", "dcb200.h")).read()
    assert re.search(r"DC_API[^;(]*\bdc_gat_bwd_edge_heads_ext\s*\(", hdr)
    assert "dc_gat_bwd_edge_heads_ext" in _abi.PROTOTYPES and hasattr(_abi.lib(), "dc_gat_bwd_edge_heads_ext")
    schema = str(torch.ops.dcb200.gat_conv_heads_backward.default._schema)
    assert "Tensor? dalpha_e=None" in schema and "Tensor? dalpha_s=None" in schema
