"""CPU tests of multi-head GATConv: the reference (the oracle for concat, tests/gat_reference.py for the mean over heads) against an
independent dense fp64 formulation per head, its symmetries, and the parameters of the drop-in layer."""
import math
import re
import os

import pytest
import torch

import oracle
from helpers import assert_close
from gat_reference import gat_reference

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _g(seed=0, n=60, e=400, f=21):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(n, f, generator=g), torch.randint(0, n, (2, e), generator=g)


def _dense_fp64(layer, x, ei):
    """Per head: softmax over the dense masked score matrix (self loop included), then concat or mean, + bias."""
    n, H, C = x.shape[0], layer.heads, layer.out_channels
    xs = (x.double() @ layer.lin.weight.double().t()).view(n, H, C)
    mask = torch.eye(n, dtype=torch.bool)
    mask[ei[1], ei[0]] = True
    outs = []
    for h in range(H):
        a_s = xs[:, h] @ layer.att_src[0, h].double()
        a_d = xs[:, h] @ layer.att_dst[0, h].double()
        e = torch.nn.functional.leaky_relu(a_d[:, None] + a_s[None, :], layer.negative_slope).masked_fill(~mask, float("-inf"))
        outs.append(torch.softmax(e, dim=1) @ xs[:, h])
    out = torch.cat(outs, 1) if layer.concat else torch.stack(outs, 0).mean(0)
    return out + layer.bias.double()


@pytest.mark.parametrize("heads", [2, 4])
@pytest.mark.parametrize("concat", [True, False])
def test_gatconv_heads_vs_dense(heads, concat):
    x, ei = _g(2)
    ei = torch.unique(ei[:, ei[0] != ei[1]], dim=1)      # dense form cannot express duplicate edges
    torch.manual_seed(2)
    layer = gat_reference(21, 8, heads=heads, concat=concat)
    with torch.no_grad():
        layer.bias.uniform_(-0.5, 0.5)
    assert layer.bias.shape == ((heads * 8,) if concat else (8,))
    out = layer(x, ei)
    assert out.shape == (x.shape[0], heads * 8 if concat else 8)
    assert_close(out, _dense_fp64(layer, x, ei).float(), what=f"GATConv H={heads} concat={concat} vs dense")


@pytest.mark.parametrize("concat", [True, False])
def test_gatconv_heads_permutation_equivariance(concat):
    x, ei = _g(3, n=200, e=1500)
    torch.manual_seed(3)
    layer = gat_reference(21, 16, heads=3, concat=concat)
    out = layer(x, ei)
    n = x.shape[0]
    perm = torch.randperm(n, generator=torch.Generator().manual_seed(0))
    inv = torch.empty_like(perm)
    inv[perm] = torch.arange(n)
    assert_close(layer(x[perm], inv[ei]), out[perm], what="permutation equivariance")


@pytest.mark.parametrize("heads", [2, 4])
def test_identical_heads_reduce_to_one_head(heads):
    """H copies of one head: the mean equals the heads=1 layer, the concat equals it tiled H times."""
    x, ei = _g(4, n=200, e=1500)
    torch.manual_seed(4)
    one = oracle.GATConv(21, 16)
    with torch.no_grad():
        one.bias.uniform_(-0.5, 0.5)
    ref = one(x, ei)
    for concat in (True, False):
        many = gat_reference(21, 16, heads=heads, concat=concat)
        with torch.no_grad():
            many.lin.weight.copy_(one.lin.weight.repeat(heads, 1))
            many.att_src.copy_(one.att_src.repeat(1, heads, 1))
            many.att_dst.copy_(one.att_dst.repeat(1, heads, 1))
            many.bias.copy_(one.bias.repeat(heads) if concat else one.bias)
        out = many(x, ei)
        assert_close(out, ref.repeat(1, heads) if concat else ref, what=f"{heads} identical heads, concat={concat}")


@pytest.mark.parametrize("heads,concat", [(1, True), (1, False), (3, True), (4, False)])
def test_layer_parameters_match_pyg(heads, concat):
    import deformcontact_b200 as dc
    torch.manual_seed(0)
    ours = dc.GATConv(21, 16, heads=heads, concat=concat)
    ref = gat_reference(21, 16, heads=heads, concat=concat)
    assert [(k, tuple(p.shape)) for k, p in ours.named_parameters()] == [(k, tuple(p.shape)) for k, p in ref.named_parameters()]
    shapes = dict((k, tuple(p.shape)) for k, p in ours.named_parameters())
    assert shapes == {"lin.weight": (heads * 16, 21), "att_src": (1, heads, 16), "att_dst": (1, heads, 16),
                      "bias": (heads * 16 if concat else 16,)}
    ours.load_state_dict(ref.state_dict())
    # glorot bounds: sqrt(6 / (fan_in + fan_out)) over the last two axes; the bias starts at zero
    assert ours.lin.weight.abs().max() <= math.sqrt(6.0 / (21 + heads * 16))
    for att in (dc.GATConv(21, 16, heads=heads, concat=concat).att_src, dc.GATConv(21, 16, heads=heads, concat=concat).att_dst):
        assert att.abs().max() <= math.sqrt(6.0 / (heads + 16))
    assert torch.equal(dc.GATConv(21, 16, heads=heads, concat=concat).bias, torch.zeros(shapes["bias"]))
    assert dc.GATConv(21, 16, heads=heads, bias=False).bias is None


def test_layer_rejects_bad_heads_and_unsupported_options():
    import deformcontact_b200 as dc
    for h in (0, -2):
        with pytest.raises(ValueError):
            dc.GATConv(21, 16, heads=h)
    for kw in (dict(dropout=0.6), dict(add_self_loops=False), dict(edge_dim=3), dict(fill_value="add")):
        with pytest.raises(NotImplementedError):
            dc.GATConv(21, 16, heads=2, **kw)


def test_multi_head_entry_points_are_declared_and_bound():
    from deformcontact_b200 import _abi
    hdr = open(os.path.join(ROOT, "include", "dcb200.h")).read()
    for name in ("dc_gat_aggregate", "dc_gat_bwd_edge_heads", "dc_gat_scatter_heads", "dc_gat_att_grad_workspace_bytes",
                 "dc_gat_att_grad"):
        assert re.search(r"DC_API[^;(]*\b" + name + r"\s*\(", hdr), name
        assert name in _abi.PROTOTYPES and hasattr(_abi.lib(), name), name
    # workspace of the attention-vector gradient: one [2, H*C] partial per 2048 rows
    assert _abi.lib().dc_gat_att_grad_workspace_bytes(4096, 8, 32) >= 2 * 2 * 8 * 32 * 4
