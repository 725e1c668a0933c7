"""GPU parity of multi-head GATConv (heads > 1, concat and mean; csrc/gat.cu) against the CPU oracle
(the mean over heads: tests/gat_reference.py on the oracle's helpers), fwd + bwd.

Tolerance: 1e-5 relative with the fp64 oracle as arbiter (tests/helpers.py)."""
import copy

import pytest
import torch

from helpers import assert_close, assert_close_arbiter
from gat_reference import gat_reference
from test_gpu_layers import _graphs

pytestmark = pytest.mark.gpu

CONFIGS = [(2, 16, True), (3, 5, True), (8, 32, True), (4, 64, False), (2, 7, False)]   # C = 5, 7: the scalar path


@pytest.fixture(scope="module")
def dc():
    import deformcontact_b200 as d
    return d


@pytest.fixture(scope="module")
def graphs():
    return _graphs()


def _pair(dc, fin, heads, C, concat, seed=0):
    torch.manual_seed(seed)
    ref = gat_reference(fin, C, heads=heads, concat=concat)
    with torch.no_grad():
        ref.bias.uniform_(-0.2, 0.2)
    ours = dc.GATConv(fin, C, heads=heads, concat=concat)
    ours.load_state_dict(ref.state_dict())
    return ref, ours.cuda()


def _input(x0, fin):
    if fin == x0.shape[1]:
        return x0
    return torch.randn(x0.shape[0], fin, generator=torch.Generator().manual_seed(fin))


def _run(layer, x, ei, gout, relu=False):
    """-> (out, [dx, dW, datt_src, datt_dst, dbias]) of one forward + backward."""
    xx = x.clone().requires_grad_(True)
    layer.zero_grad(set_to_none=True)
    out = layer(xx, ei, relu=relu)
    out.backward(gout)
    return out.detach().clone(), [xx.grad.clone()] + [p.grad.clone() for p in layer.parameters()]


@pytest.mark.parametrize("heads,C,concat", CONFIGS)
@pytest.mark.parametrize("graph", ["knn", "sphere", "mesh", "weird", "empty"])
@pytest.mark.parametrize("fin", [21, 256])
def test_gat_heads_forward_backward(dc, graphs, heads, C, concat, graph, fin):
    x0, ei = graphs[graph]
    x = _input(x0, fin)
    ref, ours = _pair(dc, fin, heads, C, concat)
    ref64 = copy.deepcopy(ref).double()
    xr, xo, x64 = x.clone().requires_grad_(True), x.clone().cuda().requires_grad_(True), x.double().requires_grad_(True)
    out_r, out_o, out_64 = ref(xr, ei), ours(xo, ei.cuda()), ref64(x64, ei)
    what = f"H={heads} C={C} concat={concat} {graph} fin={fin}"
    assert_close_arbiter(out_o, out_r, out_64, what=f"{what} out")
    go = torch.randn(out_r.shape, generator=torch.Generator().manual_seed(1))
    out_r.backward(go), out_o.backward(go.cuda()), out_64.backward(go.double())
    assert_close_arbiter(xo.grad, xr.grad, x64.grad, what=f"{what} dx")
    for (k, pr), (_, po), (_, p64) in zip(ref.named_parameters(), ours.named_parameters(), ref64.named_parameters()):
        assert_close_arbiter(po.grad, pr.grad, p64.grad, what=f"{what} d{k}")


@pytest.mark.parametrize("heads,C,concat", [(4, 64, True), (2, 7, False)])
def test_gat_heads_fused_relu(dc, graphs, heads, C, concat):
    x, ei = graphs["knn"]
    _, ours = _pair(dc, 21, heads, C, concat, seed=3)
    go = torch.randn(x.shape[0], heads * C if concat else C, generator=torch.Generator().manual_seed(2)).cuda()
    xa = x.clone().cuda().requires_grad_(True)
    fused = ours(xa, ei.cuda(), relu=True)
    fused.backward(go)
    ga = [xa.grad.clone()] + [p.grad.clone() for p in ours.parameters()]
    ours.zero_grad(set_to_none=True)
    xb = x.clone().cuda().requires_grad_(True)
    plain = torch.relu(ours(xb, ei.cuda()))
    plain.backward(go)
    gb = [xb.grad.clone()] + [p.grad.clone() for p in ours.parameters()]
    assert torch.equal(fused, plain)
    for a, b in zip(ga, gb):
        assert_close(a, b, what="fused relu grad")


def test_gat_heads_deterministic_across_csr_rebuilds(dc, graphs):
    x, ei = graphs["weird"]
    _, ours = _pair(dc, 21, 8, 32, True)
    go = torch.randn(x.shape[0], 256, generator=torch.Generator().manual_seed(4)).cuda()
    res = []
    for _ in range(2):
        dc.ops.clear_csr_cache()
        res.append(_run(ours, x.cuda(), ei.cuda(), go))
    assert torch.equal(res[0][0], res[1][0])
    for a, b in zip(res[0][1], res[1][1]):
        assert torch.equal(a, b)


def test_gat_heads_prebuilt_graph_csr_gives_the_same_bits(dc, graphs):
    x, ei = graphs["mesh"]
    _, ours = _pair(dc, 21, 4, 64, False)
    go = torch.randn(x.shape[0], 64, generator=torch.Generator().manual_seed(5)).cuda()
    res = []
    for prebuilt in (False, True):
        dc.ops.clear_csr_cache()
        e = dc.ops.GraphCSR(ei.cuda(), x.shape[0], "gat") if prebuilt else ei.cuda()
        res.append(_run(ours, x.cuda(), e, go, relu=True))
    assert torch.equal(res[0][0], res[1][0])
    for a, b in zip(res[0][1], res[1][1]):
        assert torch.equal(a, b)


def test_gat_heads_cuda_graph_replay_is_bit_identical(dc, graphs):
    x, ei = graphs["knn"]
    _, ours = _pair(dc, 21, 3, 5, True)
    x, ei = x.cuda(), ei.cuda()
    go = torch.randn(x.shape[0], 15, generator=torch.Generator().manual_seed(6)).cuda()
    eager = _run(ours, x, ei, go)                      # also builds both CSR structures outside the capture
    xs = x.clone().requires_grad_(True)
    ours.zero_grad(set_to_none=True)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):                         # warm-up on the capture stream
        ours(xs, ei).backward(go)
    torch.cuda.current_stream().wait_stream(s)
    ours.zero_grad(set_to_none=True)
    xs.grad = None
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out = ours(xs, ei)
        out.backward(go)
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(out, eager[0])
    for a, b in zip([xs.grad] + [p.grad for p in ours.parameters()], eager[1]):
        assert torch.equal(a, b)


def test_gat_heads_opcheck(dc, graphs):
    x, ei = graphs["knn"]
    x, ei = x.cuda(), ei.cuda()
    mk = lambda *s_: torch.randn(*s_, device="cuda", requires_grad=True)
    tu = ("test_schema", "test_faketensor")
    for heads, C, concat in [(2, 16, True), (3, 5, False)]:
        b = mk(heads * C if concat else C)
        torch.library.opcheck(torch.ops.dcb200.gat_conv_heads.default,
                              (x, ei, mk(heads * C, 21), mk(1, heads, C), mk(1, heads, C), b, 0.2, heads, concat, True, 0, None),
                              test_utils=tu)


def test_gat_heads_abi_rejects_bad_shapes_before_launch(dc):
    from deformcontact_b200 import _abi, ops
    ei = torch.tensor([[0, 1, 2], [1, 2, 0]], device="cuda")
    g = ops.GraphCSR(ei, 3, "gat")
    H, C = 2, 4
    f = lambda *s_: torch.zeros(*s_, device="cuda")
    xs, a, al_e, al_s, out = f(3, H * C), f(3, H), f(3, H), f(3, H), f(3, H * C)
    p = lambda t: t.data_ptr()
    st = torch.cuda.current_stream().cuda_stream
    rpt, nbt, eidt = g.t                               # the by-source structure is built before counting launches
    torch.cuda.synchronize()
    n0 = _abi.lib().dc_launch_count()

    def agg(h, c, ldx, ldo, xs_ptr=p(xs)):
        return ("dc_gat_aggregate", p(g.rowptr), p(g.nbr), p(g.eid), xs_ptr, ldx, p(a), p(a), 0.2, h, c, 1, None, 0, 3, p(out), ldo,
                p(al_e), p(al_s), st)
    for bad in (agg(0, C, H * C, H * C), agg(H, 0, H * C, H * C), agg(-1, C, H * C, H * C), agg(H, C, H * C - 1, H * C),
                agg(H, C, H * C, H * C - 1), agg(H, C, H * C, H * C, None)):
        with pytest.raises(_abi.DcError):
            _abi.call(*bad)
    bwd = lambda h, c, ldx, ldd: ("dc_gat_bwd_edge_heads", p(g.rowptr), p(g.nbr), p(g.eid), p(a), p(a), 0.2, p(al_e), p(al_s), p(xs),
                                  ldx, p(out), ldd, c, 1.0, h, c, 3, p(al_e), p(al_s), p(a), st)
    for bad in (bwd(0, C, H * C, H * C), bwd(H, 0, H * C, H * C), bwd(H, C, H * C - 1, H * C), bwd(H, C, H * C, H * C - 1)):
        with pytest.raises(_abi.DcError):
            _abi.call(*bad)
    sct = lambda h, c, ldd, lddx: ("dc_gat_scatter_heads", p(rpt), p(nbt), p(eidt), p(al_e), p(al_s), p(al_e), p(al_s), p(a),
                                   p(xs), p(xs), p(out), ldd, c, 1.0, h, c, 3, p(out), lddx, p(a), st)
    for bad in (sct(0, C, H * C, H * C), sct(H, 0, H * C, H * C), sct(H, C, H * C - 1, H * C), sct(H, C, H * C, H * C - 1)):
        with pytest.raises(_abi.DcError):
            _abi.call(*bad)
    ws = torch.empty(_abi.lib().dc_gat_att_grad_workspace_bytes(3, H, C), dtype=torch.uint8, device="cuda")
    att = lambda h, c, ldx: ("dc_gat_att_grad", p(xs), ldx, p(a), p(a), 3, h, c, p(out), p(out), p(ws), ws.numel(), st)
    for bad in (att(0, C, H * C), att(H, 0, H * C), att(H, C, H * C - 1)):
        with pytest.raises(_abi.DcError):
            _abi.call(*bad)
    assert _abi.lib().dc_launch_count() == n0
    _abi.call(*agg(H, C, H * C, H * C))                # the same call with good arguments launches
    torch.cuda.synchronize()
    assert _abi.lib().dc_launch_count() == n0 + 1


@pytest.mark.parametrize("slope", [1.0, 0.2])
def test_gat_heads_c3_size_vs_fp64_oracle_on_gpu(dc, slope):
    """256 graphs x 2000 nodes, kNN-8 (E = 4.1M), H = 8, C = 32, F_in = 256: against the oracle evaluated in fp64 on the GPU.

    With slope 1 leaky_relu is the identity, the layer is smooth, and the output and every gradient are held to 1e-5 of fp64,
    except datt_dst, which is then exactly 0 (a_dst[i] shifts every score of receiver i alike and the softmax ignores it): it
    must vanish to rounding, within 1e-5 of the scale of datt_src.
    With slope 0.2 the derivative of leaky_relu jumps at z = 0: among 33M (edge, head) scores a few lie within fp32 rounding of 0,
    fp32 and fp64 take different branches there, and the gradient of the nodes at both ends of such an edge (and every sum over
    nodes) moves by O(1) relative to its rounding error.  The output and dbias do not see the branch and are compared in full,
    dx on the rows that no edge with |z| < 1e-4 touches."""
    B, n, k, fin, H, C = 256, 2000, 8, 256, 8, 32
    gen = torch.Generator(device="cuda").manual_seed(0)
    pos = torch.rand(B * n, 3, generator=gen, device="cuda")
    ei = dc.knn_graph(pos, k, ptr=torch.arange(B + 1, device="cuda") * n)
    x = torch.randn(B * n, fin, generator=gen, device="cuda")
    go = torch.randn(B * n, H * C, generator=gen, device="cuda")
    torch.manual_seed(7)
    ref = gat_reference(fin, C, heads=H, concat=True, negative_slope=slope)
    with torch.no_grad():
        ref.bias.uniform_(-0.2, 0.2)
    ours = dc.GATConv(fin, C, heads=H, concat=True, negative_slope=slope)
    ours.load_state_dict(ref.state_dict())
    ours = ours.cuda()
    ref64 = copy.deepcopy(ref).double().cuda()
    x64 = x.double().requires_grad_(True)
    out_64 = ref64(x64, ei)
    out_64.backward(go.double())
    ref_all = [out_64.detach().float(), x64.grad.float()] + [p.grad.float() for p in ref64.parameters()]
    with torch.no_grad():
        xs64 = (x.double() @ ref64.lin.weight.t()).view(-1, H, C)
        a_s, a_d = (xs64 * ref64.att_src).sum(-1), (xs64 * ref64.att_dst).sum(-1)
        N = x.shape[0]
        src, dst = torch.cat([ei[0], torch.arange(N, device="cuda")]), torch.cat([ei[1], torch.arange(N, device="cuda")])
        near = ((a_s[src] + a_d[dst]).abs() < 1e-4).any(1)
        resolved = torch.ones(N, dtype=torch.bool, device="cuda")
        resolved[src[near]] = False
        resolved[dst[near]] = False
    del out_64, ref64, x64, xs64
    torch.cuda.empty_cache()
    out, grads = _run(ours, x, ei, go)
    names = ["out", "dx"] + [k_ for k_, _ in ours.named_parameters()]
    for name, a, b in zip(names, [out] + grads, ref_all):
        if slope == 1.0 and name == "att_dst":
            scale = grads[names.index("att_src") - 1].abs().max().item()
            assert b.abs().max().item() <= 1e-9 * scale and a.abs().max().item() <= 1e-5 * scale, "datt_dst must vanish"
        elif slope == 1.0 or name in ("out", "bias"):
            assert_close(a, b, what=f"C3-size {name} vs fp64")
        elif name == "dx":
            assert resolved.float().mean() > 0.99
            assert_close(a[resolved], b[resolved], what=f"C3-size dx vs fp64 on {int(resolved.sum())} of {N} rows")
