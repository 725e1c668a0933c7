"""GPU tests of GATConv's ``return_attention_weights`` (PyG 2.5.2's ``(out, (edge_index_sl, alpha))``): the forward, alpha and
every gradient against the reference (tests/gat_attention_reference.py) with fp64 as arbiter, for a loss on ``out``, on ``alpha``
and on both; bit-identity of the paths that do not use alpha; the extended by-receiver entry point; capture; opcheck; the ABI.

Tolerance: 1e-5 relative with the fp64 reference as arbiter (tests/helpers.py)."""
import copy

import pytest
import torch

from helpers import assert_close, assert_close_arbiter
from gat_attention_reference import GATConvAttention
from test_gpu_layers import _graphs

pytestmark = pytest.mark.gpu

CONFIGS = [(1, 32, True), (2, 16, True), (8, 32, True), (4, 64, False), (2, 7, False)]   # C = 7: the scalar path
LOSSES = ["out", "alpha", "both"]


@pytest.fixture(scope="module")
def dc():
    import deformcontact_b200 as d
    return d


@pytest.fixture(scope="module")
def graphs():
    return _graphs()


def _pair(dc, fin, heads, C, concat, seed=0, slope=0.2):
    torch.manual_seed(seed)
    ref = GATConvAttention(fin, C, heads=heads, concat=concat, negative_slope=slope)
    with torch.no_grad():
        ref.bias.uniform_(-0.2, 0.2)
    ours = dc.GATConv(fin, C, heads=heads, concat=concat, negative_slope=slope)
    ours.load_state_dict(ref.state_dict())
    return ref, ours.cuda()


def _input(x0, fin=21):
    """Seeded random features of width ``fin``, as test_gpu_gat_heads: the sphere graph's own 25 features are nearly the same on
    every node, and there the attention-vector gradients are sums that cancel to rounding (the fp32 oracle itself is 4e-5 from
    fp64 on them), whatever computes them."""
    if fin == x0.shape[1]:
        return x0
    return torch.randn(x0.shape[0], fin, generator=torch.Generator().manual_seed(fin))


def _backward(loss, out, alpha, go, ga):
    ts, gs = [], []
    if loss in ("out", "both"):
        ts.append(out), gs.append(go)
    if loss in ("alpha", "both"):
        ts.append(alpha), gs.append(ga)
    torch.autograd.backward(ts, gs)


def _grads(x, layer):
    return [x.grad] + [p.grad for p in layer.parameters()]


def _run(layer, x, ei, go, ga=None, loss="out", relu=False, attention=True):
    """-> (out, edge_index_sl, alpha, [dx, dW, datt_src, datt_dst, dbias]) of one forward + backward."""
    xx = x.clone().requires_grad_(True)
    layer.zero_grad(set_to_none=True)
    if attention:
        out, (ei_sl, alpha) = layer(xx, ei, relu=relu, return_attention_weights=True)
    else:
        out, ei_sl, alpha = layer(xx, ei, relu=relu), None, None
    _backward(loss, out, alpha, go, ga)
    clone = lambda t: None if t is None else t.detach().clone()
    return clone(out), ei_sl, clone(alpha), [clone(g) for g in _grads(xx, layer)]


def _same_bits(a, b):
    assert torch.equal(a[0], b[0])
    for u, v in zip(a[3], b[3]):
        assert (u is None and v is None) or torch.equal(u, v)


@pytest.mark.parametrize("loss", LOSSES)
@pytest.mark.parametrize("heads,C,concat", CONFIGS)
@pytest.mark.parametrize("graph", ["knn", "sphere", "mesh", "weird", "empty"])
def test_attention_forward_backward(dc, graphs, heads, C, concat, graph, loss):
    x, ei = graphs[graph]
    x = _input(x)
    ref, ours = _pair(dc, 21, heads, C, concat)
    ref64 = copy.deepcopy(ref).double()
    xr, xo, x64 = x.clone().requires_grad_(True), x.clone().cuda().requires_grad_(True), x.double().requires_grad_(True)
    out_r, (ei_r, al_r) = ref(xr, ei, return_attention_weights=True)
    out_o, (ei_o, al_o) = ours(xo, ei.cuda(), return_attention_weights=True)
    out_64, (_, al_64) = ref64(x64, ei, return_attention_weights=True)
    what = f"H={heads} C={C} concat={concat} {graph} loss={loss}"
    assert ei_o.dtype == torch.int64 and ei_o.device == xo.device and torch.equal(ei_o.cpu(), ei_r), f"{what} edge_index_sl"
    assert al_o.dtype == torch.float32 and al_o.shape == (ei_r.shape[1], heads), f"{what} alpha shape"
    assert_close_arbiter(out_o, out_r, out_64, what=f"{what} out")
    assert_close_arbiter(al_o, al_r, al_64, what=f"{what} alpha")
    go = torch.randn(out_r.shape, generator=torch.Generator().manual_seed(1))
    ga = torch.randn(al_r.shape, generator=torch.Generator().manual_seed(2))
    _backward(loss, out_r, al_r, go, ga)
    _backward(loss, out_o, al_o, go.cuda(), ga.cuda())
    _backward(loss, out_64, al_64, go.double(), ga.double())
    assert_close_arbiter(xo.grad, xr.grad, x64.grad, what=f"{what} dx")
    for (k, pr), (_, po), (_, p64) in zip(ref.named_parameters(), ours.named_parameters(), ref64.named_parameters()):
        if pr.grad is None:          # the bias does not reach alpha: no gradient, as in PyG
            assert loss == "alpha" and k == "bias" and po.grad is None, f"{what} d{k}"
            continue
        assert_close_arbiter(po.grad, pr.grad, p64.grad, what=f"{what} d{k}")


@pytest.mark.parametrize("heads,C,concat", [c for c in CONFIGS if c[0] > 1])
def test_out_and_its_gradients_are_unchanged_by_requesting_alpha(dc, graphs, heads, C, concat):
    x, ei = graphs["weird"]
    _, ours = _pair(dc, 21, heads, C, concat, seed=1)
    x, ei = x.cuda(), ei.cuda()
    go = torch.randn(x.shape[0], heads * C if concat else C, generator=torch.Generator().manual_seed(3)).cuda()
    _same_bits(_run(ours, x, ei, go, attention=False), _run(ours, x, ei, go))


def test_one_head_out_with_alpha_is_within_tolerance_of_the_default_path(dc, graphs):
    """Two fp32 kernels, each within rounding of fp64: the multi-head path taken with alpha is held to the default heads = 1 path
    with the fp64 reference as arbiter."""
    x, ei = graphs["knn"]
    ref, ours = _pair(dc, 21, 1, 32, True, seed=2)
    go = torch.randn(x.shape[0], 32, generator=torch.Generator().manual_seed(4))
    ref64 = copy.deepcopy(ref).double()
    x64 = x.double().requires_grad_(True)
    out_64 = ref64(x64, ei)
    out_64.backward(go.double())
    a, b = _run(ours, x.cuda(), ei.cuda(), go.cuda(), attention=False), _run(ours, x.cuda(), ei.cuda(), go.cuda())
    assert_close_arbiter(b[0], a[0], out_64, what="H=1 out with alpha")
    for u, v, w in zip(b[3], a[3], _grads(x64, ref64)):
        assert_close_arbiter(u, v, w, what="H=1 grads with alpha")


def _bwd_inputs(dc, graphs, heads, C, concat, graph="weird"):
    from deformcontact_b200 import ops
    x, ei = graphs[graph]
    _, ours = _pair(dc, 21, heads, C, concat, seed=5)
    x, ei = x.cuda(), ei.cuda()
    with torch.no_grad():
        out, xs, a_src, a_dst, alpha_e, alpha_s = torch.ops.dcb200.gat_conv_heads(
            x, ei, ours.lin.weight, ours.att_src, ours.att_dst, ours.bias, 0.2, heads, concat, False, 0, None)
    g = ops.graph_csr(ei, x.shape[0], "gat")
    dout = torch.randn(out.shape, generator=torch.Generator(device="cuda").manual_seed(6), device="cuda")
    return ops, g, (a_src, a_dst, alpha_e, alpha_s, xs, dout)


@pytest.mark.parametrize("heads,C,concat", [(1, 32, True), (8, 32, True), (2, 7, False)])
def test_extended_entry_point_with_null_or_zero_dalpha_gives_the_same_bits(dc, graphs, heads, C, concat):
    from deformcontact_b200 import _abi
    ops, g, (a_src, a_dst, alpha_e, alpha_s, xs, dout) = _bwd_inputs(dc, graphs, heads, C, concat)
    hs, scale = ops._dout_heads(heads, C, concat)
    p = lambda t: None if t is None else t.data_ptr()
    st = torch.cuda.current_stream().cuda_stream

    def run(name, *dalpha):
        res = (torch.zeros_like(alpha_e), torch.empty_like(alpha_s), torch.empty_like(alpha_s))
        _abi.call(name, p(g.rowptr), p(g.nbr), p(g.eid), p(a_src), p(a_dst), 0.2, p(alpha_e), p(alpha_s), p(xs), xs.stride(0), p(dout),
                  dout.stride(0), hs, scale, heads, C, g.N, *[p(t) for t in dalpha], *[p(t) for t in res], st)
        return res
    base = run("dc_gat_bwd_edge_heads")
    for dalpha in ((None, None), (torch.zeros_like(alpha_e), torch.zeros_like(alpha_s)), (torch.zeros_like(alpha_e), None)):
        for a, b in zip(base, run("dc_gat_bwd_edge_heads_ext", *dalpha)):
            assert torch.equal(a, b)


def test_extended_entry_point_adds_dalpha(dc, graphs):
    """dz of (dout, dalpha) = dz of (dout + dalpha-only): the receiver pass is linear in its gradient inputs."""
    ops, g, (a_src, a_dst, alpha_e, alpha_s, xs, dout) = _bwd_inputs(dc, graphs, 4, 64, False)
    gen = torch.Generator(device="cuda").manual_seed(7)
    de, ds = torch.randn(alpha_e.shape, generator=gen, device="cuda"), torch.randn(alpha_s.shape, generator=gen, device="cuda")
    args = (g, a_src, a_dst, 0.2, alpha_e, alpha_s, xs)
    both = ops.gat_bwd_edge_heads(*args, dout, 4, 64, False, de, ds)
    only_out = ops.gat_bwd_edge_heads(*args, dout, 4, 64, False)
    only_alpha = ops.gat_bwd_edge_heads(*args, torch.zeros_like(dout), 4, 64, False, de, ds)
    for a, b, c in zip(both, only_out, only_alpha):
        assert_close(a, b + c, what="dz linear in (dout, dalpha)")


def test_fused_relu_applies_to_out_only(dc, graphs):
    x, ei = graphs["knn"]
    _, ours = _pair(dc, 21, 4, 64, True, seed=3)
    x, ei = x.cuda(), ei.cuda()
    go = torch.randn(x.shape[0], 256, generator=torch.Generator().manual_seed(2)).cuda()
    xa = x.clone().requires_grad_(True)
    fused, (_, al_f) = ours(xa, ei, relu=True, return_attention_weights=True)
    ga = torch.randn(al_f.shape, generator=torch.Generator().manual_seed(3)).cuda()
    torch.autograd.backward([fused, al_f], [go, ga])
    gf = [t.clone() for t in _grads(xa, ours)]
    ours.zero_grad(set_to_none=True)
    xb = x.clone().requires_grad_(True)
    plain, (_, al_p) = ours(xb, ei, return_attention_weights=True)
    torch.autograd.backward([torch.relu(plain), al_p], [go, ga])
    assert torch.equal(fused, torch.relu(plain)) and torch.equal(al_f, al_p)
    for a, b in zip(gf, _grads(xb, ours)):
        assert_close(a, b, what="fused relu grad")


def test_prebuilt_graph_csr_and_csr_rebuilds_give_the_same_bits(dc, graphs):
    x, ei = graphs["weird"]
    _, ours = _pair(dc, 21, 8, 32, True)
    x, ei = x.cuda(), ei.cuda()
    go = torch.randn(x.shape[0], 256, generator=torch.Generator().manual_seed(4)).cuda()
    ga = torch.randn(int((ei[0] != ei[1]).sum()) + x.shape[0], 8, generator=torch.Generator().manual_seed(5)).cuda()
    res = []
    for prebuilt in (False, False, True):
        dc.ops.clear_csr_cache()
        e = dc.ops.GraphCSR(ei, x.shape[0], "gat") if prebuilt else ei
        res.append(_run(ours, x, e, go, ga, loss="both", relu=True))
    for r in res[1:]:
        _same_bits(res[0], r)
        assert torch.equal(r[1], res[0][1]) and torch.equal(r[2], res[0][2])


def test_cuda_graph_capture_with_a_loss_on_alpha(dc, graphs):
    x, ei = graphs["mesh"]
    _, ours = _pair(dc, 21, 2, 7, False, seed=6)
    x, ei = x.cuda(), ei.cuda()
    go = torch.randn(x.shape[0], 7, generator=torch.Generator().manual_seed(6)).cuda()
    ga = torch.randn(int((ei[0] != ei[1]).sum()) + x.shape[0], 2, generator=torch.Generator().manual_seed(7)).cuda()
    eager = _run(ours, x, ei, go, ga, loss="both")       # builds the structures and the attention edges outside the capture
    xs = x.clone().requires_grad_(True)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):                           # warm-up on the capture stream
        out, (_, alpha) = ours(xs, ei, return_attention_weights=True)
        torch.autograd.backward([out, alpha], [go, ga])
    torch.cuda.current_stream().wait_stream(s)
    ours.zero_grad(set_to_none=True)
    xs.grad = None
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out, (ei_sl, alpha) = ours(xs, ei, return_attention_weights=True)
        torch.autograd.backward([out, alpha], [go, ga])
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(out, eager[0]) and torch.equal(alpha, eager[2]) and torch.equal(ei_sl, eager[1])
    for a, b in zip(_grads(xs, ours), eager[3]):
        assert torch.equal(a, b)


def test_opcheck_of_the_backward_with_dalpha(dc, graphs):
    x, ei = graphs["weird"]
    x, ei = x.cuda(), ei.cuda()
    E, N = ei.shape[1], x.shape[0]
    mk = lambda *s_: torch.randn(*s_, device="cuda")
    tu = ("test_schema", "test_faketensor")
    for heads, C, concat in [(1, 32, True), (3, 5, False)]:
        w, a_s, a_d, b = mk(heads * C, 21), mk(1, heads, C), mk(1, heads, C), mk(heads * C if concat else C)
        fwd = (x, ei, w, a_s, a_d, b, 0.2, heads, concat, True, 0, None)
        torch.library.opcheck(torch.ops.dcb200.gat_conv_heads.default, fwd, test_utils=tu)
        out, xs, asrc, adst, al_e, al_s = torch.ops.dcb200.gat_conv_heads(*fwd)
        for de, ds in ((None, None), (mk(E, heads), mk(N, heads)), (None, mk(N, heads))):
            torch.library.opcheck(torch.ops.dcb200.gat_conv_heads_backward.default,
                                  (mk(*out.shape), out, x, ei, w, a_s, a_d, xs, asrc, adst, al_e, al_s, 0.2, heads, concat, True, 0,
                                   None, True, True, de, ds), test_utils=tu)


def test_extended_entry_point_rejects_bad_arguments_before_launch(dc):
    from deformcontact_b200 import _abi, ops
    ei = torch.tensor([[0, 1, 2], [1, 2, 0]], device="cuda")
    g = ops.GraphCSR(ei, 3, "gat")
    H, C = 2, 4
    f = lambda *s_: torch.zeros(*s_, device="cuda")
    xs, a, al_e, al_s, out, dz_e, dz_s, da = f(3, H * C), f(3, H), f(3, H), f(3, H), f(3, H * C), f(3, H), f(3, H), f(3, H)
    p = lambda t: t.data_ptr()
    st = torch.cuda.current_stream().cuda_stream
    torch.cuda.synchronize()
    n0 = _abi.lib().dc_launch_count()

    def ext(h, c, ldx, ldd, dout=p(out), rowptr=p(g.rowptr), dz=p(dz_e)):
        return ("dc_gat_bwd_edge_heads_ext", rowptr, p(g.nbr), p(g.eid), p(a), p(a), 0.2, p(al_e), p(al_s), p(xs), ldx, dout, ldd, c,
                1.0, h, c, 3, p(al_e), p(al_s), dz, p(dz_s), p(da), st)
    for bad in (ext(0, C, H * C, H * C), ext(-1, C, H * C, H * C), ext(H, 0, H * C, H * C), ext(H, C, H * C - 1, H * C),
                ext(H, C, H * C, H * C - 1), ext(H, C, H * C, H * C, dout=None), ext(H, C, H * C, H * C, rowptr=None),
                ext(H, C, H * C, H * C, dz=None)):
        with pytest.raises(_abi.DcError):
            _abi.call(*bad)
    assert _abi.lib().dc_launch_count() == n0
    _abi.call(*ext(H, C, H * C, H * C))                 # the same call with good arguments launches
    torch.cuda.synchronize()
    assert _abi.lib().dc_launch_count() == n0 + 1


def test_c3_size_loss_on_out_and_alpha_vs_fp64_on_gpu(dc):
    """256 graphs x 2000 nodes, kNN-8 (E = 4.1M), H = 8, C = 32, F_in = 256, a loss on out and alpha: against the reference in
    fp64 on the GPU.  Slope 1 keeps the layer smooth (see test_gpu_gat_heads: with slope 0.2 a few of the 37M scores sit within
    rounding of the leaky-ReLU kink).  alpha does not depend on a_dst (it shifts every score of a receiver alike), so datt_dst
    must vanish to rounding, within 1e-5 of the scale of datt_src."""
    B, n, k, fin, H, C = 256, 2000, 8, 256, 8, 32
    gen = torch.Generator(device="cuda").manual_seed(0)
    pos = torch.rand(B * n, 3, generator=gen, device="cuda")
    ei = dc.knn_graph(pos, k, ptr=torch.arange(B + 1, device="cuda") * n)
    x = torch.randn(B * n, fin, generator=gen, device="cuda")
    go = torch.randn(B * n, H * C, generator=gen, device="cuda")
    ga = torch.randn(ei.shape[1] + B * n, H, generator=gen, device="cuda")        # kNN without loops: E_nl = E
    ref, ours = _pair(dc, fin, H, C, True, seed=7, slope=1.0)
    ref64 = copy.deepcopy(ref).double().cuda()
    x64 = x.double().requires_grad_(True)
    out_64, (ei_64, al_64) = ref64(x64, ei, return_attention_weights=True)
    torch.autograd.backward([out_64, al_64], [go.double(), ga.double()])
    ref_all = [out_64.detach().float(), al_64.detach().float(), x64.grad.float()] + [p.grad.float() for p in ref64.parameters()]
    del out_64, al_64, ref64, x64
    torch.cuda.empty_cache()
    out, ei_sl, alpha, grads = _run(ours, x, ei, go, ga, loss="both")
    assert torch.equal(ei_sl, ei_64)
    names = ["out", "alpha", "dx"] + [k_ for k_, _ in ours.named_parameters()]
    for name, a, b in zip(names, [out, alpha] + grads, ref_all):
        if name == "att_dst":
            scale = grads[names.index("att_src") - 2].abs().max().item()
            assert b.abs().max().item() <= 1e-9 * scale and a.abs().max().item() <= 1e-5 * scale, "datt_dst must vanish"
        else:
            assert_close(a, b, what=f"C3-size {name} vs fp64")
