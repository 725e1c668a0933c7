"""Full-size (BASELINE.json configs) checks through size-independent properties: linearity, adjointness, permutation
equivariance, determinism and agreement with an fp64 evaluation on a random sample of rows.  These complement, not replace,
oracle parity at full size: run on the GPU, the oracle is fast enough at C3 (tests/test_gpu_c3_shapes.py compares the step,
its K1 hops and its K2 products with it there)."""
import pytest
import torch

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def dc():
    import deformcontact_b200 as d
    return d


def _big_knn_batch(dc, n_graphs, n_nodes, k, seed=0):
    g = torch.Generator(device="cuda").manual_seed(seed)
    pos = torch.rand(n_graphs * n_nodes, 3, generator=g, device="cuda") - 0.5
    ptr = torch.arange(n_graphs + 1, device="cuda") * n_nodes
    ei = dc.knn_graph(pos, k, ptr=ptr)
    return pos, ei


def test_c2_size_hop_properties(dc):
    B, n, k, F = 64, 5000, 8, 256
    pos, ei = _big_knn_batch(dc, B, n, k)
    N = B * n
    assert ei.shape[1] == N * k
    # block-diagonal: no edge crosses graphs; in-degree == k
    assert torch.equal(ei[0] // n, ei[1] // n)
    assert torch.equal(torch.bincount(ei[1], minlength=N), torch.full((N,), k, device="cuda"))
    G = dc.ops.GraphCSR(ei, N, "tag")
    g = torch.Generator(device="cuda").manual_seed(1)
    a = torch.randn(N, F, generator=g, device="cuda")
    b = torch.randn(N, F, generator=g, device="cuda")
    ha, hb = dc.ops.spmm(G.rowptr, G.nbr, a, dis=G.dis), dc.ops.spmm(G.rowptr, G.nbr, b, dis=G.dis)
    hab = dc.ops.spmm(G.rowptr, G.nbr, a + 2 * b, dis=G.dis)
    assert (hab - (ha + 2 * hb)).abs().max() <= 1e-5 * hab.abs().max()          # linearity
    assert torch.equal(ha, dc.ops.spmm(G.rowptr, G.nbr, a, dis=G.dis))           # determinism
    # adjointness <A h, g> == <h, A^T g> in fp64
    rp, nb, _ = G.t
    gt = dc.ops.spmm(rp, nb, b, dis=G.dis)
    lhs = (ha.double() * b.double()).sum()
    rhs = (a.double() * gt.double()).sum()
    assert abs(lhs - rhs) <= 1e-6 * abs(lhs)
    # sampled rows against an fp64 evaluation of the definition
    rows = torch.randint(0, N, (256,), generator=g, device="cuda")
    deg = torch.bincount(ei[1], minlength=N).double()
    dis = deg.pow(-0.5)
    for i in rows.tolist()[:64]:
        m = ei[1] == i
        ref = (dis[ei[0][m]].unsqueeze(1) * dis[i] * a[ei[0][m]].double()).sum(0)
        assert (ha[i].double() - ref).abs().max() <= 1e-5 * ref.abs().max()


def test_c4_single_large_mesh_knn_and_layers(dc):
    N, k = 200_000, 16
    pos, ei = _big_knn_batch(dc, 1, N, k, seed=3)
    assert ei.shape == (2, N * k)
    # sortedness / structure properties of the kNN result
    assert torch.equal(ei[1], torch.arange(N, device="cuda").repeat_interleave(k))
    assert (ei[0] != ei[1]).all()
    d = (pos[ei[0]] - pos[ei[1]]).square().sum(1).view(N, k)
    assert (d[:, 1:] >= d[:, :-1] * (1 - 1e-5)).all()                             # ascending per query (torch's own rounding of d)
    # exactness on sampled queries against a brute-force fp64 ranking
    g = torch.Generator(device="cuda").manual_seed(0)
    for q in torch.randint(0, N, (16,), generator=g, device="cuda").tolist():
        dd = (pos.double() - pos[q].double()).square().sum(1)
        dd[q] = float("inf")
        ref = torch.topk(dd, k, largest=False).indices.sort().values
        assert torch.equal(ei[0].view(N, k)[q].sort().values, ref)
    layer = dc.TAGConv(21, 64).cuda()
    x = dc.to_log_freq(pos)
    out = layer(x, ei, relu=True)
    assert out.shape == (N, 64) and torch.isfinite(out).all()


def test_permutation_equivariance_full_layer(dc):
    B, n, k = 8, 2000, 8
    pos, ei = _big_knn_batch(dc, B, n, k, seed=7)
    N = B * n
    layer = dc.TAGConv(21, 256).cuda()
    x = dc.to_log_freq(pos)
    out = layer(x, ei)
    perm = torch.randperm(N, device="cuda")
    inv = torch.empty_like(perm)
    inv[perm] = torch.arange(N, device="cuda")
    out_p = layer(x[perm], inv[ei])
    assert (out_p - out[perm]).abs().max() <= 1e-5 * out.abs().max()
