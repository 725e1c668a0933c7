"""CPU checks of the edge-weight reference (tests/edge_weight_reference.py) and of the layers' edge_weight argument.

The reference is checked against an independent dense fp64 formulation, against the oracle's unweighted layers (all-ones
weights give the same bits) and on the self-loop rule of ``add_remaining_self_loops``."""
import copy

import pytest
import torch

import oracle
from oracle import convs
from edge_weight_reference import GCNConvWeighted, TAGConvWeighted, dense_adjacency_fp64, gcn_norm_weighted, last_loop_edge


def _graph(seed=0, n=40, e=200):
    g = torch.Generator().manual_seed(seed)
    ei = torch.randint(0, n - 4, (2, e), generator=g)                          # duplicates, random loops, isolated tail nodes
    ei = torch.cat([ei, torch.tensor([[3, 5, 3, 7], [3, 5, 3, 7]])], 1)      # duplicate loops on node 3
    w = torch.empty(ei.shape[1]).uniform_(0.1, 2.0, generator=g)
    x = torch.randn(n, 6, generator=g)
    return x, ei, w


@pytest.mark.parametrize("normalize", [True, False])
def test_tag_reference_matches_dense_fp64(normalize):
    x, ei, w = _graph()
    torch.manual_seed(0)
    ref = TAGConvWeighted(6, 5, normalize=normalize).double()
    w64 = w.double().requires_grad_(True)
    out = ref(x.double(), ei, w64)
    A = dense_adjacency_fp64(ei, w64, x.shape[0], normalize=normalize)
    h, dense = x.double(), x.double() @ ref.lins[0].weight.t()
    for lin in ref.lins[1:]:
        h = A @ h
        dense = dense + h @ lin.weight.t()
    dense = dense + ref.bias
    assert torch.allclose(out, dense, rtol=1e-12, atol=1e-12)
    go = torch.randn(out.shape, generator=torch.Generator().manual_seed(1), dtype=torch.float64)
    g_ref, = torch.autograd.grad(out, w64, go)
    g_dense, = torch.autograd.grad(dense, w64, go)
    assert torch.allclose(g_ref, g_dense, rtol=1e-10, atol=1e-12)


@pytest.mark.parametrize("improved", [False, True])
def test_gcn_reference_matches_dense_fp64(improved):
    x, ei, w = _graph(1)
    torch.manual_seed(0)
    ref = GCNConvWeighted(6, 5, improved=improved).double()
    w64 = w.double().requires_grad_(True)
    out = ref(x.double(), ei, w64)
    A = dense_adjacency_fp64(ei, w64, x.shape[0], add_self_loops=True, fill_value=2.0 if improved else 1.0)
    dense = A @ (x.double() @ ref.lin.weight.t()) + ref.bias
    assert torch.allclose(out, dense, rtol=1e-12, atol=1e-12)
    go = torch.randn(out.shape, generator=torch.Generator().manual_seed(1), dtype=torch.float64)
    g_ref, = torch.autograd.grad(out, w64, go)
    g_dense, = torch.autograd.grad(dense, w64, go)
    assert torch.allclose(g_ref, g_dense, rtol=1e-10, atol=1e-12)


def test_all_ones_weights_give_the_oracle_bits():
    x, ei, _ = _graph(2)
    ones = torch.ones(ei.shape[1])
    for add in (False, True):
        e_ref, w_ref = convs.gcn_norm(ei, x.shape[0], add)
        e_w, w_w = gcn_norm_weighted(ei, ones, x.shape[0], add)
        assert torch.equal(e_ref, e_w) and torch.equal(w_ref, w_w)
    for normalize in (True, False):
        torch.manual_seed(3)
        plain = oracle.TAGConv(6, 5, normalize=normalize)
        weighted = TAGConvWeighted(6, 5, normalize=normalize)
        weighted.load_state_dict(plain.state_dict())
        assert torch.equal(plain(x, ei), weighted(x, ei, ones))
    torch.manual_seed(4)
    plain, weighted = oracle.GCNConv(6, 5), GCNConvWeighted(6, 5)
    weighted.load_state_dict(plain.state_dict())
    assert torch.equal(plain(x, ei), weighted(x, ei, ones))


def test_loop_rule_last_loop_edge_supplies_the_weight_and_takes_the_gradient():
    # node 0: loops at edges 1 and 3 (3 is the last); node 1: no loop (fill_value); node 2: one loop (edge 4)
    ei = torch.tensor([[1, 0, 2, 0, 2, 0], [0, 0, 1, 0, 2, 2]])
    assert last_loop_edge(ei, 3).tolist() == [3, -1, 4]
    w = torch.tensor([0.5, 0.7, 1.5, 1.3, 0.9, 1.1], dtype=torch.float64, requires_grad=True)
    for fill in (1.0, 2.0):
        e2, norm = gcn_norm_weighted(ei, w, 3, True, fill)
        assert e2.tolist() == [[1, 2, 0, 0, 1, 2], [0, 1, 2, 0, 1, 2]]     # non-loop edges in order, then one loop per node
        deg = torch.tensor([0.5 + 1.3, 1.5 + fill, 1.1 + 0.9], dtype=torch.float64)
        dis = deg.pow(-0.5)
        assert torch.allclose(norm[3:], dis * torch.tensor([1.3, fill, 0.9], dtype=torch.float64) * dis)
        g, = torch.autograd.grad(norm.sum(), w)
        assert g[1] == 0.0 and g[3] != 0.0 and g[4] != 0.0              # the superseded loop gets nothing


def test_zero_in_weight_gives_zero_degree_gradient_not_nan():
    ei = torch.tensor([[1, 2], [0, 0]])
    w = torch.tensor([0.0, 0.0], dtype=torch.float64, requires_grad=True)
    _, norm = gcn_norm_weighted(ei, w, 3)
    g, = torch.autograd.grad(norm.sum(), w)
    assert torch.equal(norm, torch.zeros(2, dtype=torch.float64)) and torch.isfinite(g).all()


def test_layer_edge_weight_validation():
    import deformcontact_b200 as dc
    from deformcontact_b200 import _abi
    x, ei = torch.randn(10, 8), torch.tensor([[0, 1, 2], [1, 2, 3]])
    for layer in (dc.TAGConv(8, 4), dc.GCNConv(8, 4)):
        with pytest.raises(TypeError):
            layer(x, ei, True)                          # an old positional relu
        with pytest.raises(TypeError):
            layer(x, ei, [1.0, 1.0, 1.0])
        with pytest.raises(_abi.DcError, match="dtype"):
            layer(x, ei, torch.ones(3, dtype=torch.float64))
        with pytest.raises(_abi.DcError, match=r"\[3\]"):
            layer(x, ei, torch.ones(4))
        with pytest.raises(_abi.DcError, match=r"\[3\]"):
            layer(x, ei, torch.ones(3, 1))
        with pytest.raises(_abi.DcError, match="CUDA"):
            layer(x, ei, torch.ones(3))


def test_gcn_constructor_options():
    import deformcontact_b200 as dc
    assert dc.GCNConv(8, 4).improved is False and dc.GCNConv(8, 4, improved=True).improved is True
    for kw in (dict(cached=True), dict(add_self_loops=False), dict(normalize=False)):
        with pytest.raises(NotImplementedError):
            dc.GCNConv(8, 4, **kw)


def test_state_dict_keys_unchanged_and_load_from_reference():
    import deformcontact_b200 as dc
    torch.manual_seed(0)
    for ref, ours in ((TAGConvWeighted(8, 4), dc.TAGConv(8, 4)), (GCNConvWeighted(8, 4, improved=True), dc.GCNConv(8, 4, improved=True)),
                      (oracle.GCNConv(8, 4), dc.GCNConv(8, 4))):
        assert list(ours.state_dict()) == list(ref.state_dict())
        ours.load_state_dict(copy.deepcopy(ref.state_dict()))
