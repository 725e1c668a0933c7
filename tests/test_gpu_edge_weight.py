"""GPU parity of TAGConv / GCNConv with PyG's edge_weight (csrc/gcn_norm.cu: the weighted norm, the SDDMM and the normalisation
backward) against tests/edge_weight_reference.py, fwd + bwd including dL/dedge_weight.

Tolerance: 1e-5 relative with the fp64 reference as arbiter (tests/helpers.py)."""
import copy

import pytest
import torch

from helpers import assert_close, assert_close_arbiter
from edge_weight_reference import GCNConvWeighted, TAGConvWeighted, gcn_norm_weighted
from oracle import convs
from test_gpu_layers import _graphs

pytestmark = pytest.mark.gpu

# (layer, option): TAGConv normalize, GCNConv improved
CONFIGS = [("TAGConv", True), ("TAGConv", False), ("GCNConv", False), ("GCNConv", True)]


@pytest.fixture(scope="module")
def dc():
    import deformcontact_b200 as d
    return d


@pytest.fixture(scope="module")
def graphs():
    return _graphs()


def _weights(ei, seed=0):
    return torch.empty(ei.shape[1]).uniform_(0.1, 2.0, generator=torch.Generator().manual_seed(seed))


def _pair(dc, layer, opt, fin, fout, seed=0):
    torch.manual_seed(seed)
    if layer == "TAGConv":
        ref, ours = TAGConvWeighted(fin, fout, normalize=opt), dc.TAGConv(fin, fout, normalize=opt)
    else:
        ref, ours = GCNConvWeighted(fin, fout, improved=opt), dc.GCNConv(fin, fout, improved=opt)
    with torch.no_grad():
        ref.bias.uniform_(-0.2, 0.2)
    ours.load_state_dict(ref.state_dict())
    return ref, ours.cuda()


def _input(x0, fin):
    return x0 if fin == x0.shape[1] else torch.randn(x0.shape[0], fin, generator=torch.Generator().manual_seed(fin))


def _run(layer, x, ei, w, go, relu=False, ptr=None, need_x=True):
    """-> (out, [dx or None, dedge_weight or None, *parameter grads]) of one forward + backward."""
    xx = x.clone().requires_grad_(need_x)
    ww = None if w is None else w.clone().requires_grad_(True)
    layer.zero_grad(set_to_none=True)
    out = layer(xx, ei, ww, relu=relu, ptr=ptr) if ww is not None else layer(xx, ei, relu=relu, ptr=ptr)
    out.backward(go)
    grads = [xx.grad.clone() if need_x else None, None if ww is None else ww.grad.clone()]
    return out.detach().clone(), grads + [p.grad.clone() for p in layer.parameters()]


@pytest.mark.parametrize("layer,opt", CONFIGS)
@pytest.mark.parametrize("graph", ["knn", "sphere", "mesh", "weird", "empty"])
@pytest.mark.parametrize("fin", [21, 256])
def test_edge_weight_forward_backward(dc, graphs, layer, opt, graph, fin):
    x0, ei = graphs[graph]
    x, w = _input(x0, fin), _weights(ei)
    ref, ours = _pair(dc, layer, opt, fin, 32)
    ref64 = copy.deepcopy(ref).double()
    xr, xo, x64 = x.clone().requires_grad_(True), x.clone().cuda().requires_grad_(True), x.double().requires_grad_(True)
    wr, wo, w64 = w.clone().requires_grad_(True), w.clone().cuda().requires_grad_(True), w.double().requires_grad_(True)
    out_r, out_o, out_64 = ref(xr, ei, wr), ours(xo, ei.cuda(), wo), ref64(x64, ei, w64)
    what = f"{layer}({opt}) {graph} fin={fin}"
    assert_close_arbiter(out_o, out_r, out_64, what=f"{what} out")
    go = torch.randn(out_r.shape, generator=torch.Generator().manual_seed(1))
    out_r.backward(go), out_o.backward(go.cuda()), out_64.backward(go.double())
    assert_close_arbiter(xo.grad, xr.grad, x64.grad, what=f"{what} dx")
    if w.numel():
        assert_close_arbiter(wo.grad, wr.grad, w64.grad, what=f"{what} dedge_weight")
    assert wo.grad.shape == w.shape
    for (k, pr), (_, po), (_, p64) in zip(ref.named_parameters(), ours.named_parameters(), ref64.named_parameters()):
        assert_close_arbiter(po.grad, pr.grad, p64.grad, what=f"{what} d{k}")
    # dedge_weight alone (the first layer's input needs no gradient): same bits as with dx
    _, grads = _run(ours, x.cuda(), ei.cuda(), w.cuda(), go.cuda(), need_x=False)
    assert torch.equal(grads[1], wo.grad)


@pytest.mark.parametrize("improved", [False, True])
def test_gcn_transposed_edge_index_with_duplicate_loops(dc, improved):
    """PyG's common ``edge_index = pairs.t()`` (strides (1, 2)) on a graph with self loops, duplicate loops on one node and a
    node without a loop: the loop weights come from the last loop edge of each node, as for a contiguous edge list."""
    g = torch.Generator().manual_seed(18)
    n = 60
    pairs = torch.randint(0, n - 5, (400, 2), generator=g)
    pairs = torch.cat([pairs, torch.tensor([[3, 3], [7, 7], [3, 3], [11, 11], [3, 3]])])    # three loops on node 3
    pairs = pairs[(pairs[:, 0] != 20) | (pairs[:, 1] != 20)]                                # and none on node 20
    ei_t = pairs.t()
    assert not ei_t.is_contiguous()
    x, w = torch.randn(n, 21, generator=g), _weights(ei_t, 19)
    ref, ours = _pair(dc, "GCNConv", improved, 21, 16, seed=19)
    ref64 = copy.deepcopy(ref).double()
    go = torch.randn(n, 16, generator=g)
    xr, wr, x64, w64 = (x.clone().requires_grad_(True), w.clone().requires_grad_(True), x.double().requires_grad_(True),
                        w.double().requires_grad_(True))
    out_r, out_64 = ref(xr, ei_t.contiguous(), wr), ref64(x64, ei_t.contiguous(), w64)
    out_r.backward(go), out_64.backward(go.double())
    dc.ops.clear_csr_cache()
    out, grads = _run(ours, x.cuda(), ei_t.cuda(), w.cuda(), go.cuda())
    what = f"GCNConv(improved={improved}) transposed edge_index"
    assert_close_arbiter(out, out_r, out_64, what=f"{what} out")
    assert_close_arbiter(grads[0], xr.grad, x64.grad, what=f"{what} dx")
    assert_close_arbiter(grads[1], wr.grad, w64.grad, what=f"{what} dedge_weight")
    dc.ops.clear_csr_cache()
    out_c, grads_c = _run(ours, x.cuda(), ei_t.contiguous().cuda(), w.cuda(), go.cuda())
    assert torch.equal(out, out_c) and all(torch.equal(a, b) for a, b in zip(grads, grads_c))


@pytest.mark.parametrize("graph", ["knn", "weird"])
def test_gcn_odd_width_takes_the_scalar_sddmm(dc, graphs, graph):
    """out_channels = 7: x W^T has 28-byte rows, so the SDDMM runs its scalar lanes (F % 4 != 0) with a column tail."""
    x, ei = graphs[graph]
    w = _weights(ei, 20)
    ref, ours = _pair(dc, "GCNConv", True, 21, 7, seed=20)
    ref64 = copy.deepcopy(ref).double()
    go = torch.randn(x.shape[0], 7, generator=torch.Generator().manual_seed(21))
    xr, wr, x64, w64 = (x.clone().requires_grad_(True), w.clone().requires_grad_(True), x.double().requires_grad_(True),
                        w.double().requires_grad_(True))
    out_r, out_64 = ref(xr, ei, wr), ref64(x64, ei, w64)
    out_r.backward(go), out_64.backward(go.double())
    out, grads = _run(ours, x.cuda(), ei.cuda(), w.cuda(), go.cuda())
    assert_close_arbiter(out, out_r, out_64, what=f"{graph} F=7 out")
    assert_close_arbiter(grads[0], xr.grad, x64.grad, what=f"{graph} F=7 dx")
    assert_close_arbiter(grads[1], wr.grad, w64.grad, what=f"{graph} F=7 dedge_weight")


@pytest.mark.parametrize("mode", ["tag", "gcn"])
def test_weighted_hop_is_bit_identical_to_the_cpu_reference(dc, graphs, mode):
    x, ei = graphs["weird"]
    w = _weights(ei, 2)
    g = dc.ops.graph_csr(ei.cuda(), x.shape[0], mode)
    v = dc.ops.weighted_view(g, w.cuda(), True, 1.0)
    e2, norm = gcn_norm_weighted(ei, w, x.shape[0], mode == "gcn")
    h = torch.randn(x.shape[0], 32, generator=torch.Generator().manual_seed(3))
    assert torch.equal(v.propagate(h.cuda()).cpu(), convs.propagate(h, e2, norm, x.shape[0]))


@pytest.mark.parametrize("layer,opt", [("TAGConv", True), ("TAGConv", False), ("GCNConv", False)])
def test_all_ones_weights_give_the_bits_of_no_weights(dc, graphs, layer, opt):
    x0, ei = graphs["knn"]
    x = _input(x0, 256)
    _, ours = _pair(dc, layer, opt, 256, 64, seed=4)
    go = torch.randn(x.shape[0], 64, generator=torch.Generator().manual_seed(5)).cuda()
    plain = _run(ours, x.cuda(), ei.cuda(), None, go, relu=True)
    ones = _run(ours, x.cuda(), ei.cuda(), torch.ones(ei.shape[1]).cuda(), go, relu=True)
    assert torch.equal(plain[0], ones[0])
    for i, (a, b) in enumerate(zip(plain[1], ones[1])):
        if i != 1:
            assert torch.equal(a, b)


@pytest.mark.parametrize("layer,opt", CONFIGS)
def test_zero_weights_are_deleted_edges(dc, graphs, layer, opt):
    x, ei = graphs["mesh"]
    w = _weights(ei, 6)
    w[::3] = 0.0
    keep = w != 0
    _, ours = _pair(dc, layer, opt, 21, 16, seed=6)
    with torch.no_grad():
        a = ours(x.cuda(), ei.cuda(), w.cuda())
        b = ours(x.cuda(), ei[:, keep].contiguous().cuda(), w[keep].contiguous().cuda())
    assert torch.equal(a, b)


@pytest.mark.parametrize("layer,opt", CONFIGS)
@pytest.mark.parametrize("with_ptr", [False, True])
def test_deterministic_across_csr_rebuilds_and_prebuilt_graph_csr(dc, layer, opt, with_ptr):
    from deformcontact_b200 import synthetic
    rest, _, _ = synthetic.make_batch(4, 300, 8)
    x, ei = rest.x.cuda(), rest.edge_index.cuda()
    ptr = rest.ptr.tolist() if with_ptr else None
    w = _weights(ei, 7).cuda()
    _, ours = _pair(dc, layer, opt, 21, 32, seed=7)
    go = torch.randn(x.shape[0], 32, generator=torch.Generator().manual_seed(8)).cuda()
    res = []
    for prebuilt in (False, False, True):
        dc.ops.clear_csr_cache()
        e = dc.ops.GraphCSR(ei, x.shape[0], "tag" if layer == "TAGConv" else "gcn", ptr) if prebuilt else ei
        res.append(_run(ours, x, e, w, go, ptr=ptr))
    for r in res[1:]:
        assert torch.equal(res[0][0], r[0])
        for a, b in zip(res[0][1], r[1]):
            assert torch.equal(a, b)


def test_relabelled_large_cloud(dc):
    gen = torch.Generator(device="cuda").manual_seed(9)
    pos = torch.rand(40000, 3, generator=gen, device="cuda")
    ei = dc.knn_graph(pos, 8)
    x = torch.randn(40000, 32, generator=gen, device="cuda")
    w = torch.rand(ei.shape[1], generator=gen, device="cuda") * 1.9 + 0.1
    assert dc.ops.graph_csr(ei, 40000, "tag").order is not None, "the cloud must be relabelled"
    go = torch.randn(40000, 32, generator=gen, device="cuda")
    for layer, opt in [("TAGConv", True), ("GCNConv", True)]:
        ref, ours = _pair(dc, layer, opt, 32, 32, seed=10)
        out, grads = _run(ours, x, ei, w, go)
        ref = ref.double().cuda()                      # fp64 reference on the GPU
        xr, wr = x.double().requires_grad_(True), w.double().requires_grad_(True)
        out_r = ref(xr, ei, wr)
        out_r.backward(go.double())
        assert_close(out, out_r, what=f"{layer} relabelled out")
        assert_close(grads[0], xr.grad, what=f"{layer} relabelled dx")
        assert_close(grads[1], wr.grad, what=f"{layer} relabelled dedge_weight")


@pytest.mark.parametrize("layer", ["TAGConv", "GCNConv"])
@pytest.mark.parametrize("big", [False, True])
def test_layer_stack_with_weights_equals_the_plain_loop(dc, layer, big):
    if big:
        gen = torch.Generator(device="cuda").manual_seed(11)
        pos = torch.rand(33000, 3, generator=gen, device="cuda")
        ei = dc.knn_graph(pos, 8)
        x = torch.randn(33000, 32, generator=gen, device="cuda")
    else:
        x0, ei0 = _graphs()["knn"]
        x, ei = _input(x0, 32).cuda(), ei0.cuda()
    w = torch.rand(ei.shape[1], generator=torch.Generator(device="cuda").manual_seed(12), device="cuda") + 0.1
    torch.manual_seed(13)
    layers = torch.nn.ModuleList([getattr(dc, layer)(32, 32) for _ in range(3)]).cuda()
    a = dc.layers.layer_stack(layers, x, ei, edge_weight=w)
    b = x
    for conv in layers:
        b = conv(b, ei, w, relu=True)
    assert torch.equal(a, b)


@pytest.mark.parametrize("layer,opt", [("TAGConv", True), ("GCNConv", True)])
def test_cuda_graph_replay_is_bit_identical(dc, graphs, layer, opt):
    x, ei = graphs["knn"]
    x, ei = x.cuda(), ei.cuda()
    w = _weights(ei, 14).cuda()
    _, ours = _pair(dc, layer, opt, 21, 16, seed=14)
    go = torch.randn(x.shape[0], 16, generator=torch.Generator().manual_seed(15)).cuda()
    eager = _run(ours, x, ei, w, go)
    xs, ws = x.clone().requires_grad_(True), w.clone().requires_grad_(True)
    ours.zero_grad(set_to_none=True)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        ours(xs, ei, ws).backward(go)
    torch.cuda.current_stream().wait_stream(s)
    ours.zero_grad(set_to_none=True)
    xs.grad, ws.grad = None, None
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out = ours(xs, ei, ws)
        out.backward(go)
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(out, eager[0])
    for a, b in zip([xs.grad, ws.grad] + [p.grad for p in ours.parameters()], eager[1]):
        assert torch.equal(a, b)


def test_opcheck(dc, graphs):
    x, ei = graphs["knn"]
    x, ei = x.cuda(), ei.cuda()
    mk = lambda *s_: torch.randn(*s_, device="cuda", requires_grad=True)
    w = (torch.rand(ei.shape[1], device="cuda") + 0.1).requires_grad_(True)
    xp = torch.nn.functional.pad(x, (0, 11)).requires_grad_(True)       # 32 columns, as TAGConv pads 21
    tu = ("test_schema", "test_faketensor", "test_autograd_registration")
    for normalize in (True, False):
        torch.library.opcheck(torch.ops.dcb200.tag_conv_weighted.default,
                              (xp, ei, w, [mk(16, 32) for _ in range(4)], mk(16), True, normalize, 0, None), test_utils=tu)
    for fill in (1.0, 2.0):
        torch.library.opcheck(torch.ops.dcb200.gcn_conv_weighted.default, (x, ei, w, mk(16, 21), mk(16), False, fill, 0, None),
                              test_utils=tu)


@pytest.mark.parametrize("layer", ["TAGConv", "GCNConv"])
def test_no_sddmm_launch_without_weight_gradient(dc, graphs, layer):
    from deformcontact_b200 import _abi
    x, ei = graphs["knn"]
    x, ei = x.cuda(), ei.cuda()
    w = _weights(ei, 16).cuda()
    _, ours = _pair(dc, layer, True, 21, 16, seed=16)
    go = torch.randn(x.shape[0], 16, device="cuda")
    counts = []
    for need in (False, True):
        ww = w.clone().requires_grad_(need)
        xx = x.clone().requires_grad_(True)
        ours(xx, ei, ww).backward(go)               # warm (structures built)
        torch.cuda.synchronize()
        n0 = _abi.lib().dc_launch_count()
        ours(xx, ei, ww).backward(go)
        torch.cuda.synchronize()
        counts.append(_abi.lib().dc_launch_count() - n0)
    assert counts[1] == counts[0] + 2, counts       # the SDDMM and the normalisation backward, nothing else


def test_abi_rejects_bad_arguments_before_launch(dc):
    from deformcontact_b200 import _abi, ops
    ei = torch.tensor([[0, 1, 2, 2], [1, 2, 0, 2]], device="cuda")
    g = ops.graph_csr(ei, 3, "gcn")
    rpt, nbt, eidt = g.t
    f = lambda *s_: torch.zeros(*s_, device="cuda")
    w, h, s, n = f(4), f(3, 8), f(4), f(3)
    li = torch.zeros(3, dtype=torch.int32, device="cuda")
    rec = torch.zeros(4, 2, dtype=torch.int32, device="cuda")
    p = lambda t: None if t is None else t.data_ptr()
    st = torch.cuda.current_stream().cuda_stream
    torch.cuda.synchronize()
    n0 = _abi.lib().dc_launch_count()

    def norm(N=3, E=4, wt=w, loop=1, rp=g.rowptr, d=n):
        return ("dc_gcn_norm_weighted", p(ei), E, N, p(rp), p(g.nbr), p(g.eid), p(rpt), p(nbt), p(eidt), p(wt), 1.0, 1, loop, p(d),
                p(n), p(li), p(n), p(w), p(rec), p(w), p(rec), st)
    for bad in (norm(N=-1), norm(E=-1), norm(wt=None), norm(loop=2), norm(rp=None), norm(d=None)):
        with pytest.raises(_abi.DcError):
            _abi.call(*bad)

    def sddmm(F=8, npairs=1, ld=8, hp=h, out=s, nb=g.nbr, ed=g.eid):
        arr = (_abi.SddmmPair * 5)(*[_abi.SddmmPair(p(h), ld, p(hp), ld)] * 5)
        return ("dc_edge_sddmm", p(g.rowptr), p(nb), p(ed), arr, npairs, 3, F, 0, p(out), p(n), st)
    for bad in (sddmm(F=0), sddmm(npairs=0), sddmm(npairs=5), sddmm(ld=7), sddmm(hp=None), sddmm(out=None), sddmm(nb=None),
                sddmm(ed=None)):
        with pytest.raises(_abi.DcError):
            _abi.call(*bad)

    def bwd(N=3, d=n, sv=s):
        return ("dc_gcn_norm_weighted_backward", p(g.rowptr), p(g.nbr), p(g.eid), p(rpt), p(nbt), p(eidt), p(w), p(d), p(n), p(li),
                p(sv), p(n), N, 4, p(w), st)
    for bad in (bwd(N=-1), bwd(d=None), bwd(sv=None)):
        with pytest.raises(_abi.DcError):
            _abi.call(*bad)
    assert _abi.lib().dc_launch_count() == n0
    _abi.call(*sddmm())                          # the same call with good arguments launches
    torch.cuda.synchronize()
    assert _abi.lib().dc_launch_count() == n0 + 1


def test_c5_size_tagconv_with_weights_vs_fp64(dc):
    """256 graphs x 2000 nodes, kNN-8 (E = 4.1M), TAGConv(256, 256) with weights U(0.1, 2) requiring grad: output and every
    gradient, dedge_weight included, within 1e-5 of the reference evaluated in fp64 on the GPU."""
    B, n, k, F = 256, 2000, 8, 256
    gen = torch.Generator(device="cuda").manual_seed(0)
    pos = torch.rand(B * n, 3, generator=gen, device="cuda")
    ptr = torch.arange(B + 1, device="cuda") * n
    ei = dc.knn_graph(pos, k, ptr=ptr)
    x = torch.randn(B * n, F, generator=gen, device="cuda")
    w = torch.rand(ei.shape[1], generator=gen, device="cuda") * 1.9 + 0.1
    go = torch.randn(B * n, F, generator=gen, device="cuda")
    torch.manual_seed(17)
    ref = TAGConvWeighted(F, F)
    with torch.no_grad():
        ref.bias.uniform_(-0.2, 0.2)
    ours = dc.TAGConv(F, F)
    ours.load_state_dict(ref.state_dict())
    ours = ours.cuda()
    ref64 = ref.double().cuda()
    x64, w64 = x.double().requires_grad_(True), w.double().requires_grad_(True)
    out_64 = ref64(x64, ei, w64)
    out_64.backward(go.double())
    ref_all = [out_64.detach().float(), x64.grad.float(), w64.grad.float()] + [p.grad.float() for p in ref64.parameters()]
    del out_64, ref64, x64, w64
    torch.cuda.empty_cache()
    out, grads = _run(ours, x, ei, w, go, ptr=ptr.tolist())
    names = ["out", "dx", "dedge_weight"] + [k_ for k_, _ in ours.named_parameters()]
    for name, a, b in zip(names, [out] + grads, ref_all):
        assert_close(a, b, what=f"C5-size {name} vs fp64")
