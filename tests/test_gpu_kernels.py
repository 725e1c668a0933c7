"""GPU parity tests for the individual kernels (through the C ABI) against the CPU oracle."""
import pytest
import torch

import oracle
from oracle import convs as oconvs
from helpers import assert_close, canonical

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def dc():
    import deformcontact_b200 as d
    assert torch.cuda.is_available()
    return d


def _rand_graph(n, e, seed, self_loops=True, dup=True):
    g = torch.Generator().manual_seed(seed)
    ei = torch.randint(0, n, (2, e), generator=g)
    if not self_loops:
        ei = ei[:, ei[0] != ei[1]]
    if dup and ei.shape[1] > 4:
        ei = torch.cat([ei, ei[:, :3]], 1)
    return ei


def _ref_csr(ei, n, by, drop):
    e = ei.shape[1]
    key = ei[0] if by else ei[1]
    other = ei[1] if by else ei[0]
    eid = torch.arange(e)
    if drop:
        m = ei[0] != ei[1]
        key, other, eid = key[m], other[m], eid[m]
    order = torch.sort(key, stable=True).indices
    rowptr = torch.zeros(n + 1, dtype=torch.long)
    rowptr[1:] = torch.bincount(key, minlength=n).cumsum(0)
    return rowptr, other[order], eid[order]


@pytest.mark.parametrize("n,e", [(1, 0), (5, 0), (7, 20), (1000, 8000), (2049, 2048), (70001, 300017), (300, 100000),
                                 (512000, 4096000)])   # last: the C3 step's soft graph (256 x 2000 nodes, kNN-8)
@pytest.mark.parametrize("by", [0, 1])
@pytest.mark.parametrize("drop", [False, True])
def test_csr_build(dc, n, e, by, drop):
    ei = _rand_graph(n, e, seed=n + e, dup=e > 0) if e else torch.zeros(2, 0, dtype=torch.long)
    rp, nbr, eid = dc.ops.csr_build(ei.cuda(), n, by, drop)
    rrp, rnbr, reid = _ref_csr(ei, n, by, drop)
    assert torch.equal(rp.cpu().long(), rrp)
    m = int(rrp[-1])
    assert torch.equal(nbr.cpu().long()[:m], rnbr)
    assert torch.equal(eid.cpu().long()[:m], reid)


def test_csr_hub_and_isolated(dc):
    # star graph: one receiver with 50k in-edges, many isolated nodes
    n = 60000
    src = torch.arange(1, 50001)
    ei = torch.stack([src, torch.zeros_like(src)])
    rp, nbr, eid = dc.ops.csr_build(ei.cuda(), n, 0, False)
    assert int(rp[1]) == 50000 and int(rp[-1]) == 50000
    assert torch.equal(nbr.cpu().long(), src)
    dis = dc.ops.deg_inv_sqrt(rp, n).cpu()
    assert dis[1] == 0 and torch.isfinite(dis).all()
    assert dis[0] == (torch.tensor(50000.0).sqrt().reciprocal())


@pytest.mark.parametrize("F", [1, 3, 21, 24, 25, 32, 64, 100, 128, 256, 512])
@pytest.mark.parametrize("transpose", [False, True])
def test_spmm_vs_oracle_propagate(dc, F, transpose):
    n, e = 3000, 24000
    ei = _rand_graph(n, e, seed=F)
    g = torch.Generator().manual_seed(F)
    h = torch.randn(n, F, generator=g)
    _, w = oconvs.gcn_norm(ei, n, False)
    G = dc.ops.GraphCSR(ei.cuda(), n, "tag")
    if not transpose:
        ref = oconvs.propagate(h, ei, w, n)
        out = dc.ops.spmm(G.rowptr, G.nbr, h.cuda(), dis=G.dis)
    else:
        ref = oconvs.propagate(h, ei.flip(0), w, n)  # A_hat^T h
        rp, nb, _ = G.t
        out = dc.ops.spmm(rp, nb, h.cuda(), dis=G.dis)
    assert_close(out, ref, what=f"spmm F={F} T={transpose}")
    # same summation order and rounding as the CPU reference => expected bit-exact
    assert torch.equal(out.cpu(), ref), "spmm is expected to be bit-identical to the CPU scatter order"
    out2 = dc.ops.spmm(G.rowptr if not transpose else G.t[0], G.nbr if not transpose else G.t[1], h.cuda(), dis=G.dis)
    assert torch.equal(out, out2), "run-to-run determinism"


@pytest.mark.parametrize("F", [4, 24, 28, 32, 64, 100, 256, 260])
@pytest.mark.parametrize("mode", ["tag", "gcn"])
@pytest.mark.parametrize("tiles", ["graphs", "fixed"])
@pytest.mark.parametrize("variant", ["tiled", "tiled_prefetch", "smem", "lean", "blocks", "auto"])
def test_spmm_tiled_bit_identical_to_generic(dc, F, mode, tiles, variant, monkeypatch):
    """K1 v2 (tile x slice) == K1 v1 (generic) bit for bit, and both == oracle order."""
    sizes = [300, 1, 2500, 40, 7000, 900]
    n = sum(sizes)
    g = torch.Generator().manual_seed(F)
    eis, off = [], 0
    for s in sizes:
        e = torch.randint(0, s, (2, 9 * s), generator=g) + off
        eis.append(e)
        off += s
    ei = torch.cat(eis, 1)
    ptr = [0]
    for s in sizes:
        ptr.append(ptr[-1] + s)
    h = torch.randn(n, F, generator=g).cuda()
    add = torch.randn(n, F, generator=g).cuda()
    bias = torch.randn(F, generator=g).cuda()
    G = dc.ops.GraphCSR(ei.cuda(), n, mode, ptr if tiles == "graphs" else None)
    monkeypatch.setattr(dc.ops, "K1_VARIANT", variant)
    for tr in (False, True):
        rp, nb, _ = G.t if tr else (G.rowptr, G.nbr, G.eid)
        v1 = dc.ops.spmm(rp, nb, h, dis=G.dis, add=add, self_loop=(mode == "gcn"), bias=bias, relu=True)
        v2 = G.propagate(h, transpose=tr, add=add, bias=bias, relu=True)
        assert torch.equal(v1, v2)
        v1 = dc.ops.spmm(rp, nb, h, dis=G.dis, self_loop=(mode == "gcn"))
        v2 = G.propagate(h, transpose=tr)
        assert torch.equal(v1, v2)
    if mode == "tag":
        _, w = oconvs.gcn_norm(ei, n, False)
        assert torch.equal(G.propagate(h).cpu(), oconvs.propagate(h.cpu(), ei, w, n))


@pytest.mark.parametrize("variant,flags", [("blocks", 0), ("blocks", 1), ("blocks", 2), ("blocks", 3), ("blocks", 4), ("blocks", 5),
                                           ("blocks", 7), ("blocks", 8), ("blocks", 13), ("blocks", 23), ("blocks", 28), ("blocks", 61)])
@pytest.mark.parametrize("mode", ["tag", "gcn"])
def test_spmm_blocks_ragged_and_deep_rows(dc, variant, flags, mode, monkeypatch):
    """K1 v7 (edge blocks): rows deeper than the 64-edge block depth, isolated receivers, duplicate edges, self
    loops, tiles that are not multiples of 4/256 — bit-identical to the generic kernel in every launch mode."""
    g = torch.Generator().manual_seed(flags)
    sizes = [5, 1, 1031, 3, 700, 258]
    n = sum(sizes)
    ptr = [0]
    for s in sizes:
        ptr.append(ptr[-1] + s)
    eis = []
    for lo, hi in zip(ptr[:-1], ptr[1:]):
        s = hi - lo
        eis.append(torch.randint(0, s, (2, 5 * s), generator=g) + lo)
    hub = ptr[2] + 7                                  # 300 in-edges and 200 out-edges on one node (deg > 64)
    eis.append(torch.stack([torch.randint(ptr[2], ptr[3], (300,), generator=g), torch.full((300,), hub)]))
    eis.append(torch.stack([torch.full((200,), hub), torch.randint(ptr[2], ptr[3], (200,), generator=g)]))
    eis.append(torch.tensor([[hub, hub, ptr[4]], [hub, hub, ptr[4]]]))   # self loops (one duplicated)
    ei = torch.cat(eis, 1)
    ei = ei[:, torch.randperm(ei.shape[1], generator=g)]
    F = 72
    h = torch.randn(n, F, generator=g).cuda()
    add = torch.randn(n, F, generator=g).cuda()
    bias = torch.randn(F, generator=g).cuda()
    G = dc.ops.GraphCSR(ei.cuda(), n, mode, ptr)
    monkeypatch.setattr(dc.ops, "K1_VARIANT", variant)
    monkeypatch.setattr(dc.ops, "K1_FLAGS", flags)
    unit = 4
    for tr in (False, True):
        rp, nb, _ = G.t if tr else (G.rowptr, G.nbr, G.eid)
        v1 = dc.ops.spmm(rp, nb, h, dis=G.dis, add=add, self_loop=(mode == "gcn"), bias=bias, relu=True)
        v2 = G.propagate(h, transpose=tr, add=add, bias=bias, relu=True)
        assert torch.equal(v1, v2)
        v1 = dc.ops.spmm(rp, nb, h, dis=G.dis, self_loop=(mode == "gcn"))
        v2 = G.propagate(h, transpose=tr)
        assert torch.equal(v1, v2)
        assert int(G.blocks(tr, unit).status.item()) == 0
    Gf = dc.ops.GraphCSR(ei.cuda(), n, mode, None)    # fixed tiles
    assert torch.equal(Gf.propagate(h), G.propagate(h))
    # tiles that cut through graphs: sources outside the tile take the checked path
    cut = dc.ops.EdgeBlocks(G.rowptr, G.edges, n, G.edges.shape[0], [0, 500, 1037, 1500, n], unit)
    fn = dc.ops.spmm_blocks
    sw = G.self_w if mode == "gcn" else None
    assert torch.equal(fn(cut, G.rowptr, G.edges, sw, h, self_loop=(mode == "gcn")), G.propagate(h))
    assert int(cut.status.item()) == 0
    # empty graph / no edges
    G0 = dc.ops.GraphCSR(torch.zeros(2, 0, dtype=torch.long).cuda(), 10, mode)
    x0 = torch.randn(10, 8, generator=g).cuda()
    assert torch.equal(G0.propagate(x0), dc.ops.spmm(G0.rowptr, G0.nbr, x0, dis=G0.dis, self_loop=(mode == "gcn")))


def test_make_tiles():
    from deformcontact_b200.ops import make_tiles
    assert make_tiles([0, 2000, 4000, 6000], 6000) == [0, 2000, 4000, 6000]
    t = make_tiles([0, 762, 1524, 2286, 3048, 3810], 3810)
    assert t[0] == 0 and t[-1] == 3810 and all(b - a <= 2560 for a, b in zip(t, t[1:]))
    t = make_tiles([0, 200000], 200000)
    assert t[0] == 0 and t[-1] == 200000 and all(0 < b - a <= 2560 for a, b in zip(t, t[1:]))
    assert make_tiles(None, 10) is None


def test_spmm_add_bias_relu_strided(dc):
    n, e, F = 1500, 9000, 64
    ei = _rand_graph(n, e, 5)
    g = torch.Generator().manual_seed(1)
    big = torch.randn(n, 3 * F, generator=g).cuda()
    h = big[:, F:2 * F]
    add = torch.randn(n, F, generator=g).cuda()
    bias = torch.randn(F, generator=g).cuda()
    G = dc.ops.GraphCSR(ei.cuda(), n, "tag")
    out = torch.zeros(n, 2 * F).cuda()
    dc.ops.spmm(G.rowptr, G.nbr, h, dis=G.dis, add=add, bias=bias, relu=True, out=out[:, F:])
    _, w = oconvs.gcn_norm(ei, n, False)
    ref = torch.relu(add.cpu() + oconvs.propagate(h.cpu(), ei, w, n) + bias.cpu())
    assert_close(out[:, F:], ref, what="spmm add/bias/relu")
    assert torch.count_nonzero(out[:, :F]) == 0


@pytest.mark.parametrize("M,N,K,ta,tb", [(300, 256, 84, 0, 1), (1000, 256, 1024, 0, 1), (513, 21, 256, 0, 0),
                                         (256, 21, 5000, 1, 0), (256, 256, 40000, 1, 0), (1, 1, 1, 0, 1),
                                         (129, 130, 17, 1, 1), (2, 64, 3000, 1, 0)])
def test_gemm_simt(dc, M, N, K, ta, tb):
    g = torch.Generator().manual_seed(M + N + K)
    A = torch.randn((K, M) if ta else (M, K), generator=g)
    B = torch.randn((N, K) if tb else (K, N), generator=g)
    bias = torch.randn(N, generator=g)
    ref = ((A.t() if ta else A).double() @ (B.t() if tb else B).double() + bias.double())
    out = dc.ops.gemm([(A.cuda(), B.cuda())], M, N, bool(ta), bool(tb), bias=bias.cuda(), precision=dc.ops.GEMM_FP32)
    assert_close(out, ref.float(), what="gemm")
    out_r = dc.ops.gemm([(A.cuda(), B.cuda())], M, N, bool(ta), bool(tb), bias=bias.cuda(), relu=True,
                        precision=dc.ops.GEMM_FP32)
    assert_close(out_r, ref.clamp_min(0).float(), what="gemm relu")
    out2 = dc.ops.gemm([(A.cuda(), B.cuda())], M, N, bool(ta), bool(tb), bias=bias.cuda(), precision=dc.ops.GEMM_FP32)
    assert torch.equal(out, out2)


def test_gemm_segments_and_accumulate(dc):
    g = torch.Generator().manual_seed(0)
    M, N = 700, 256
    As = [torch.randn(M, k, generator=g) for k in (21, 21, 21, 21)]
    Bs = [torch.randn(N, k, generator=g) for k in (21, 21, 21, 21)]
    ref = sum(a.double() @ b.double().t() for a, b in zip(As, Bs))
    out = dc.ops.gemm([(a.cuda(), b.cuda()) for a, b in zip(As, Bs)], M, N, False, True, precision=dc.ops.GEMM_FP32)
    assert_close(out, ref.float(), what="4-seg gemm")
    dc.ops.gemm([(As[0].cuda(), Bs[0].cuda())], M, N, False, True, out=out, accumulate=True, precision=dc.ops.GEMM_FP32)
    assert_close(out, (ref + As[0].double() @ Bs[0].double().t()).float(), what="accumulate")


def test_colsum_relu_bwd(dc):
    g = torch.Generator().manual_seed(2)
    X = torch.randn(10007, 257, generator=g)
    assert_close(dc.ops.colsum(X.cuda()), X.double().sum(0).float(), what="colsum")
    Y = torch.randn(1000, 33, generator=g)
    dY = torch.randn(1000, 33, generator=g)
    assert torch.equal(dc.ops.relu_bwd(Y.cuda(), dY.cuda()).cpu(), dY * (Y > 0))


@pytest.mark.parametrize("n,k", [(1, 3), (3, 5), (50, 8), (1000, 8), (3000, 16), (2500, 40), (1200, 100)])
def test_knn_bit_exact(dc, n, k):
    g = torch.Generator().manual_seed(n * 31 + k)
    pos = torch.rand(n, 3, generator=g) - 0.5
    ref = oracle.knn_graph(pos, k)
    out = dc.knn_graph(pos.cuda(), k)
    assert out.dtype == torch.int64 and out.shape[0] == 2
    assert torch.equal(canonical(out), canonical(ref))
    # neighbour order inside a query is also ascending (distance, index) — compare un-sorted too
    assert torch.equal(out.cpu(), ref)


def test_knn_ties_duplicates_and_batch(dc):
    g = torch.Generator().manual_seed(3)
    pos = (torch.randint(0, 4, (600, 3), generator=g).float()) * 0.25  # lattice: many exact ties and duplicates
    batch = torch.arange(3).repeat_interleave(200)
    for b in (None, batch):
        ref = oracle.knn_graph(pos, 6, b)
        out = dc.knn_graph(pos.cuda(), 6, None if b is None else b.cuda())
        assert torch.equal(canonical(out), canonical(ref))
    ref = oracle.knn_graph(pos, 6, batch, loop=True)
    out = dc.knn_graph(pos.cuda(), 6, batch.cuda(), loop=True)
    assert torch.equal(canonical(out), canonical(ref))


def test_knn_ragged_batch(dc):
    g = torch.Generator().manual_seed(4)
    sizes = [1, 7, 300, 2, 33, 1500]
    pos = torch.rand(sum(sizes), 3, generator=g)
    batch = torch.repeat_interleave(torch.arange(len(sizes)), torch.tensor(sizes))
    ref = oracle.knn_graph(pos, 8, batch)
    out = dc.knn_graph(pos.cuda(), 8, batch.cuda())
    assert torch.equal(out.cpu(), ref)


@pytest.mark.parametrize("r,mx", [(0.05, 32), (0.15, 32), (0.3, 32), (0.2, 4), (0.5, 64)])
def test_radius_bit_exact(dc, r, mx):
    g = torch.Generator().manual_seed(int(r * 100) + mx)
    pos = torch.rand(1500, 3, generator=g)
    batch = torch.repeat_interleave(torch.arange(3), torch.tensor([400, 100, 1000]))
    for b in (None, batch):
        ref = oracle.radius_graph(pos, r, b, max_num_neighbors=mx)
        out = dc.radius_graph(pos.cuda(), r, None if b is None else b.cuda(), max_num_neighbors=mx)
        assert torch.equal(canonical(out), canonical(ref))
        assert torch.equal(out.cpu(), ref)


def test_construct_graph_reference_api(dc):
    pos = torch.rand(500, 3, generator=torch.Generator().manual_seed(9))
    assert torch.equal(dc.construct_graph(pos.cuda(), k=5).cpu(), oracle.construct_graph(pos, k=5))
    assert torch.equal(dc.construct_graph(pos.cuda(), radius=0.15).cpu(), oracle.construct_graph(pos, radius=0.15))


def test_mesh_to_graph_and_posenc(dc, golden_dir):
    v, t = oracle.uv_sphere(0.05, 20, (0.1, -0.2, 0.3))
    ref = oracle.mesh_to_graph(v, t)
    out = dc.mesh_to_graph(v, t)
    assert torch.equal(out.edge_index.cpu(), ref.edge_index)
    assert torch.equal(out.pos.cpu(), ref.pos)
    assert_close(out.x, ref.x, tol=2e-6, what="posenc")
    gold = torch.load(f"{golden_dir}/posenc.pt")
    assert_close(dc.to_log_freq(gold["pos"].cuda(), 3, 1), gold["out"], tol=2e-6, what="posenc vs reference golden")


def test_abi_errors(dc):
    from deformcontact_b200 import _abi
    with pytest.raises(_abi.DcError):
        dc.ops.csr_build(torch.zeros(2, 3, dtype=torch.long), 4)          # CPU tensor: no CPU path
    with pytest.raises(_abi.DcError):
        dc.ops.spmm(None, None, torch.zeros(4, 4).cuda())                 # null rowptr -> DC_EINVAL
    with pytest.raises(_abi.DcError):
        dc.ops.knn_table(torch.zeros(10, 3).cuda(), 500)                  # k too large -> DC_ENOSUP


@pytest.mark.parametrize("M,N,Ks,tb", [(128, 256, [32], True), (300, 64, [32, 64], True), (1000, 256, [256] * 4, True),
                                       (5000, 128, [96], False), (129, 16, [64], True), (40000, 256, [256], False)])
def test_gemm_tcgen05_3xtf32(dc, M, N, Ks, tb):
    """tcgen05 kind::tf32 GEMM with the 3-term split: fp32-class accuracy (<= 1e-5 vs fp64)."""
    g = torch.Generator().manual_seed(M + N)
    As = [torch.randn(M, k, generator=g).cuda() for k in Ks]
    Bs = [(torch.randn(N, k, generator=g) if tb else torch.randn(k, N, generator=g)).cuda() for k in Ks]
    bias = torch.randn(N, generator=g).cuda()
    ref = sum(a.double() @ (w.double().t() if tb else w.double()) for a, w in zip(As, Bs)) + bias.double()
    out = dc.ops.gemm(list(zip(As, Bs)), M, N, False, tb, bias=bias, precision=dc.ops.GEMM_TF32X3)
    assert_close(out, ref.float(), what="tcgen05 gemm")
    out_r = dc.ops.gemm(list(zip(As, Bs)), M, N, False, tb, bias=bias, relu=True, precision=dc.ops.GEMM_TF32X3)
    assert_close(out_r, ref.clamp_min(0).float(), what="tcgen05 gemm relu")
    assert torch.equal(out, dc.ops.gemm(list(zip(As, Bs)), M, N, False, tb, bias=bias, precision=dc.ops.GEMM_TF32X3))
    acc = out.clone()
    dc.ops.gemm(list(zip(As, Bs)), M, N, False, tb, out=acc, accumulate=True, precision=dc.ops.GEMM_TF32X3)
    assert_close(acc, (2 * ref - bias.double()).float(), what="tcgen05 gemm accumulate")
    # strided output view
    big = torch.zeros(M, N + 64).cuda()
    dc.ops.gemm(list(zip(As, Bs)), M, N, False, tb, bias=bias, out=big[:, 32:32 + N], precision=dc.ops.GEMM_TF32X3)
    assert torch.equal(big[:, 32:32 + N], out) and big[:, :32].abs().sum() == 0 and big[:, 32 + N:].abs().sum() == 0


def test_gemm_tc_unsupported_reports_enosup(dc):
    from deformcontact_b200 import _abi
    A, B = torch.randn(64, 21).cuda(), torch.randn(32, 21).cuda()
    with pytest.raises(_abi.DcError):
        dc.ops.gemm([(A, B)], 64, 32, False, True, precision=dc.ops.GEMM_TF32X3)     # K % 32 != 0
    out = dc.ops.gemm([(A, B)], 64, 32, False, True, precision=dc.ops.GEMM_PREFER_TC)  # falls back to fp32
    assert_close(out, (A.double() @ B.double().t()).float(), what="prefer_tc fallback")


@pytest.mark.parametrize("K,M,N", [(32, 128, 32), (333, 128, 32), (1000, 256, 256), (5000, 200, 64), (70001, 256, 256),
                                   (4096, 21, 256), (100000, 256, 32)])
def test_gemm_tcgen05_weight_gradient(dc, K, M, N):
    """K3: C = A^T B over a long contraction, MN-major tf32 operands (SWIZZLE_128B_BASE32B), chunked split-K."""
    g = torch.Generator().manual_seed(K + M + N)
    A = torch.randn(K, M, generator=g).cuda()
    B = torch.randn(K, N, generator=g).cuda()
    if M % 4:   # lda must be a multiple of 4 floats for TMA: take a view of a padded buffer
        Ap = torch.zeros(K, M + (4 - M % 4)).cuda()
        Ap[:, :M] = A
        A = Ap[:, :M]
    ref = A.double().t() @ B.double()
    out = dc.ops.gemm([(A, B)], M, N, True, False, precision=dc.ops.GEMM_TF32X3)
    assert_close(out, ref.float(), what="tcgen05 dW gemm")
    assert torch.equal(out, dc.ops.gemm([(A, B)], M, N, True, False, precision=dc.ops.GEMM_TF32X3))   # deterministic
    acc = out.clone()
    dc.ops.gemm([(A, B)], M, N, True, False, out=acc, accumulate=True, precision=dc.ops.GEMM_TF32X3)
    assert_close(acc, (2 * ref).float(), what="tcgen05 dW gemm accumulate")


@pytest.mark.parametrize("stream", [0, 1])
@pytest.mark.parametrize("F", [32, 256])
def test_hop_chain_bit_identical_to_single_hops(dc, F, stream, monkeypatch):
    """K1 v9 (L1 chain) and K1 v11 (dc_spmm_stream: per-group edge streams, rolling gather window): the hops of a layer in
    one launch == one launch per hop == generic kernel, bit for bit (forward and transposed with in-place addends), ragged
    block-diagonal batch with isolated nodes, deep rows and an empty graph."""
    from deformcontact_b200 import ops
    monkeypatch.setattr(ops, "K1_STREAM", stream)
    sizes = [700, 0, 1, 1300, 64]
    ptr = [0]
    for s_ in sizes:
        ptr.append(ptr[-1] + s_)
    N = ptr[-1]
    gen = torch.Generator().manual_seed(5)
    eis = []
    for lo, hi in zip(ptr[:-1], ptr[1:]):
        n = hi - lo
        if n == 0:
            continue
        e = torch.randint(0, n, (2, 9 * n), generator=gen)
        e[1, : min(n, 200)] = 0          # one deep row (> 64 edges)
        eis.append(e + lo)
    ei = torch.cat(eis, 1).cuda()
    g = ops.GraphCSR(ei, N, "tag", ptr)
    assert g.tiles_closed
    x = torch.randn(N, F, generator=gen).cuda()
    # forward chain into the strided [N, 3F] layout TAGConv uses
    buf = torch.zeros(N, 3 * F, device="cuda")
    hs = [x] + [buf[:, i * F:(i + 1) * F] for i in range(3)]
    ops.spmm_chain(g.rowptr, g.edges, None, [(hs[i], None, hs[i + 1]) for i in range(3)], tile_ptr=g.tile_ptr, n_tiles=g.n_tiles)
    ref = x
    for i in range(3):
        ref = ops.spmm(g.rowptr, g.nbr, ref, dis=g.dis)
        assert torch.equal(hs[i + 1], ref), f"forward hop {i}"
    # transposed chain with in-place addends
    adds = [torch.randn(N, F, generator=gen).cuda() for _ in range(3)]
    d = [a.clone() for a in adds]
    g3 = torch.randn(N, F, generator=gen).cuda()
    ops.spmm_chain(g.t[0], g._edges_t, None, [(g3, d[2], d[2]), (d[2], d[1], d[1]), (d[1], d[0], d[0])], tile_ptr=g.tile_ptr,
                   n_tiles=g.n_tiles)
    ref = g3
    for i in (2, 1, 0):
        ref = ops.spmm(g.t[0], g.t[1], ref, dis=g.dis, add=adds[i])
        assert torch.equal(d[i], ref), f"transposed hop {i}"
    # propagate_chain falls back to single hops when a graph is split across tiles (tiles not closed)
    big = ops.GraphCSR(ei, N, "tag", [0, N])
    if not big.tiles_closed:
        out = [torch.empty(N, F, device="cuda") for _ in range(2)]
        ops.propagate_chain(big, [(x, None, out[0]), (out[0], None, out[1])])
        assert torch.equal(out[0], hs[1])


def test_hop_chain_rejects_bad_args(dc):
    from deformcontact_b200 import ops, _abi
    ei = torch.randint(0, 100, (2, 500)).cuda()
    g = ops.GraphCSR(ei, 100, "tag", [0, 100])
    x = torch.randn(100, 24).cuda()
    with pytest.raises(_abi.DcError):      # F % 32 != 0 (the L1 chain kernel; dc_spmm_stage takes any F % 4 == 0)
        ops.spmm_chain(g.rowptr, g.edges, None, [(x, None, torch.empty_like(x))], tile_ptr=g.tile_ptr, n_tiles=g.n_tiles)
    x = torch.randn(100, 32).cuda()
    with pytest.raises(_abi.DcError):      # in aliases out
        ops.spmm_chain(g.rowptr, g.edges, None, [(x, None, x)], tile_ptr=g.tile_ptr, n_tiles=g.n_tiles)


def test_stream_chain_rejects_bad_args(dc, monkeypatch):
    """dc_spmm_stream keeps the contract of dc_spmm_chain: F % 32 == 0, in != out; and self loops (GCN) never reach it."""
    from deformcontact_b200 import ops, _abi
    monkeypatch.setattr(ops, "K1_STREAM", 1)
    ei = torch.randint(0, 100, (2, 500)).cuda()
    g = ops.GraphCSR(ei, 100, "tag", [0, 100])
    x = torch.randn(100, 24).cuda()
    with pytest.raises(_abi.DcError):
        ops.spmm_chain(g.rowptr, g.edges, None, [(x, None, torch.empty_like(x))], tile_ptr=g.tile_ptr, n_tiles=g.n_tiles)
    x = torch.randn(100, 32).cuda()
    with pytest.raises(_abi.DcError):
        ops.spmm_chain(g.rowptr, g.edges, None, [(x, None, x)], tile_ptr=g.tile_ptr, n_tiles=g.n_tiles)
    gg = ops.GraphCSR(ei, 100, "gcn", [0, 100])     # self loops: falls through to the v9 kernel, same numbers as single hops
    out = torch.empty_like(x)
    ops.spmm_chain(gg.rowptr, gg.edges, gg.self_w, [(x, None, out)], self_loop=True, tile_ptr=gg.tile_ptr, n_tiles=gg.n_tiles)
    assert torch.equal(out, gg.propagate(x))


def _clouds():
    g = torch.Generator().manual_seed(77)
    uni = torch.rand(6000, 3, generator=g) - 0.5
    clustered = torch.cat([0.01 * torch.randn(2500, 3, generator=g) + 0.3, 0.02 * torch.randn(2500, 3, generator=g) - 0.2,
                           torch.rand(300, 3, generator=g)])
    dup = torch.rand(700, 3, generator=g)
    dup = torch.cat([dup, dup[:400], dup[:100]])               # exact duplicates: ties on the distance -> lower index wins
    planar = torch.cat([torch.rand(4000, 2, generator=g), torch.zeros(4000, 1)], 1)
    lattice = torch.stack(torch.meshgrid(*[torch.arange(16.0)] * 3, indexing="ij"), -1).reshape(-1, 3) * 0.25   # massive ties
    same = torch.full((300, 3), 0.125)
    shifted = torch.rand(3000, 3, generator=g) * 1e-3 + 100.0   # tiny extent far from the origin (coarse fp32 grid)
    return dict(uniform=uni, clustered=clustered, duplicates=dup, planar=planar, lattice=lattice, coincident=same, shifted=shifted)


@pytest.mark.parametrize("name", ["uniform", "clustered", "duplicates", "planar", "lattice", "coincident", "shifted"])
def test_grid_search_bit_identical_to_brute_force(dc, name):
    """K4g (uniform grid) == K4 (tiled brute force) bit for bit: neighbour tables incl. order, for kNN (several k, loop)
    and radius search (incl. truncation to the lowest indices), on uniform / clustered / degenerate clouds."""
    from deformcontact_b200 import ops
    pos = _clouds()[name].cuda()
    ext = float((pos.max(0).values - pos.min(0).values).max())
    try:
        for k, loop in ((16, False), (8, True), (40, False), (100, False)):
            ops.KNN_MODE = "brute"
            ref = ops.knn_table(pos, k, loop=loop)
            ops.KNN_MODE = "grid"
            out = ops.knn_table(pos, k, loop=loop)
            assert torch.equal(out, ref), f"knn {name} k={k} loop={loop}: {(out != ref).sum().item()} entries differ"
        for r, mx, loop in ((0.05 * ext + 1e-6, 32, False), (0.2 * ext + 1e-6, 5, False), (0.1 * ext + 1e-6, 64, True), (0.0, 8, False)):
            ops.KNN_MODE = "brute"
            ref, rc = ops.radius_table(pos, r, loop=loop, max_num_neighbors=mx)
            ops.KNN_MODE = "grid"
            out, oc = ops.radius_table(pos, r, loop=loop, max_num_neighbors=mx)
            assert torch.equal(out, ref) and torch.equal(oc, rc), f"radius {name} r={r} max={mx} loop={loop}"
    finally:
        ops.KNN_MODE = "auto"


def test_grid_search_large_cloud_vs_oracle_and_auto_dispatch(dc):
    """Above KNN_GRID_MIN points a single cloud goes to the grid automatically; edge_index equals the oracle's on a sample
    of queries (the oracle is O(N^2): checked per query against its brute-force definition) and the brute-force kernel's."""
    from deformcontact_b200 import ops
    g = torch.Generator().manual_seed(3)
    pos = torch.rand(40000, 3, generator=g)
    assert ops._use_grid(pos.shape[0], None, None, 17)
    ei = dc.knn_graph(pos.cuda(), 16)
    ops.KNN_MODE = "brute"
    try:
        ref = dc.knn_graph(pos.cuda(), 16)
    finally:
        ops.KNN_MODE = "auto"
    assert torch.equal(ei, ref)
    sub = torch.arange(0, 40000, 997)
    d = ((pos[sub, None, :] - pos[None, :, :]) ** 2)
    d2 = (d[..., 0] + d[..., 1]) + d[..., 2]                      # the oracle's association (oracle/graphs.py:_sqdist)
    d2[torch.arange(sub.numel()), sub] = float("inf")
    vals, idx = torch.sort(d2, dim=1, stable=True)
    clean = vals[:, 15] < vals[:, 16]                             # a tie at the k-th place is resolved by index: skip it here
    want = idx[:, :16].sort(1).values
    tab = ei[0].cpu().reshape(40000, 16)[sub].sort(1).values
    assert clean.sum() >= sub.numel() - 2 and torch.equal(tab[clean], want[clean])
    # a batch vector is never taken for one cloud (batches of large clouds have their own grid-per-graph entry point)
    assert not ops._use_grid(40000, torch.zeros(40000, dtype=torch.long), None, 17)


def test_batched_grid_search_bit_identical_to_brute_force(dc):
    """dc_knn_grid_batched / dc_radius_grid_batched (one grid per graph of a batch) == dc_knn / dc_radius (tiled brute force) bit for
    bit, incl. neighbour order and the radius search's truncation to the lowest indices:
    a ragged batch of uniform / clustered / degenerate clouds with an empty graph, a one-point graph and a graph with fewer
    than k points in between, and the 256 x 2000 positions of the C3 step; several k, loop on / off; through ``ptr`` and through a ``batch`` vector; auto dispatch by the
    average cloud size; the device-side hand-back of a batch a grid cannot split."""
    from deformcontact_b200 import ops
    g = torch.Generator().manual_seed(5)
    clouds = _clouds()
    tiny = [torch.zeros(0, 3), torch.rand(1, 3, generator=g), torch.rand(5, 3, generator=g)]
    stretched = torch.rand(3000, 3, generator=g) * torch.tensor([10.0, 0.1, 1.0])
    # "benign": grids split every cloud (the device-side cost estimate keeps the batch on the grid); "mixed": clustered / planar /
    # stretched clouds as well — whichever kernel the device-side decision picks, the table is the brute-force one
    benign = [clouds["uniform"], tiny[0], clouds["duplicates"], tiny[1], clouds["lattice"], tiny[2], clouds["shifted"],
              clouds["coincident"], torch.rand(5000, 3, generator=g) - 2.0]
    mixed = [clouds["uniform"], tiny[0], clouds["clustered"], tiny[1], clouds["duplicates"], tiny[2], clouds["planar"],
             clouds["lattice"], clouds["coincident"], clouds["shifted"], stretched]
    # the C3 step's soft graphs: 256 clouds of 2000 points, drawn as synthetic.make_batch draws them
    c3 = [torch.rand(2000, 3, generator=torch.Generator().manual_seed(1234 + i)) - 0.5 for i in range(256)]
    try:
        for parts, want_grid in ((benign, True), (mixed, None), (c3, True)):
            sizes = [p.shape[0] for p in parts]
            pos = torch.cat(parts).cuda()
            ptr = torch.tensor([0] + sizes).cumsum(0).cuda()
            batch = torch.repeat_interleave(torch.arange(len(sizes)), torch.tensor(sizes)).cuda()
            for k, loop in ((8, False), (16, True), (40, False), (100, False)):
                ops.KNN_MODE = "brute"
                ref = ops.knn_table(pos, k, ptr=ptr, loop=loop)
                ops.KNN_MODE = "grid"
                out = ops.knn_table(pos, k, ptr=ptr, loop=loop)
                assert torch.equal(out, ref), f"batched knn k={k} loop={loop}: {(out != ref).sum().item()} entries differ"
                if want_grid is not None:
                    assert ops.grid_took_it(out) == want_grid
                assert torch.equal(ops.knn_table(pos, k, batch=batch, loop=loop), ref)
            for r, mx, loop in ((0.05, 32, False), (0.2, 5, False), (0.1, 64, True), (0.0, 8, False), (1.0e-3, 16, False)):
                ops.KNN_MODE = "brute"
                ref, rc = ops.radius_table(pos, r, ptr=ptr, loop=loop, max_num_neighbors=mx)
                ops.KNN_MODE = "grid"
                out_r, oc = ops.radius_table(pos, r, ptr=ptr, loop=loop, max_num_neighbors=mx)
                assert torch.equal(out_r, ref) and torch.equal(oc, rc), f"batched radius r={r} max={mx} loop={loop}"
                if want_grid is not None:
                    assert ops.grid_took_it(out_r) == want_grid
        # neighbours never cross graph boundaries
        gid = batch[out.clamp(min=0).long()]
        assert bool(((gid == batch[:, None]) | (out < 0)).all())
        # auto: by the total and the average cloud size
        ops.KNN_MODE = "auto"
        big = torch.rand(8 * 3000, 3, generator=g).cuda()
        p4 = torch.arange(0, 8 * 3000 + 1, 3000).cuda()
        assert ops.grid_took_it(ops.knn_table(big, 8, ptr=p4))
        small = torch.arange(0, 8 * 3000 + 1, 120).cuda()
        t_small = ops.knn_table(big, 8, ptr=small)
        assert not ops.grid_took_it(t_small)
        assert not ops.grid_took_it(ops.knn_table(big[:6000], 8, ptr=p4[:3]))      # a small batch stays on the brute-force kernel
        ops.KNN_MODE = "grid"
        assert torch.equal(ops.knn_table(big, 8, ptr=small), t_small)
        # one graph with a far outlier: its grid is one cell -> the whole batch goes back to the brute-force kernel, same output
        bad = big.clone()
        bad[5] = 1.0e4
        out = ops.knn_table(bad, 8, ptr=p4)
        ops.KNN_MODE = "brute"
        assert torch.equal(out, ops.knn_table(bad, 8, ptr=p4))
        assert not ops.grid_took_it(out)
    finally:
        ops.KNN_MODE = "auto"


def test_grid_search_hands_unsplittable_clouds_to_brute_force(dc):
    """Device-side dispatch of K4g: one far outlier puts the whole cloud into one cell -> the brute-force kernel runs (no
    performance cliff), a uniform cloud stays on the grid; the output is the same either way."""
    from deformcontact_b200 import ops
    g = torch.Generator().manual_seed(12)
    uni = torch.rand(20000, 3, generator=g)
    outlier = torch.cat([uni, torch.tensor([[1.0e4, 1.0e4, 1.0e4]])])
    try:
        for pos, want_grid in ((uni.cuda(), True), (outlier.cuda(), False)):
            ops.KNN_MODE = "brute"
            ref = ops.knn_table(pos, 16)
            ops.KNN_MODE = "grid"
            out = ops.knn_table(pos, 16)
            assert torch.equal(out, ref)
            assert ops.grid_took_it(out) == want_grid
    finally:
        ops.KNN_MODE = "auto"


@pytest.mark.parametrize("F,graph_nodes", [(256, 2000), (256, 1500), (24, 2000), (28, 762), (64, 2900), (128, 3500), (36, 700)])
def test_staged_hop_chain_bit_identical_to_single_hops(dc, F, graph_nodes):
    """K1 v10 (dc_spmm_stage: tile slice staged in shared memory by TMA, 4..8 float4 lanes per receiver depending on the
    tile size, any F % 4 == 0) == one generic launch per hop, bit for bit — forward chain into the strided [N, 3F] layout and
    transposed chain with in-place addends; ragged batch with a deep row, isolated nodes, an empty and a one-node graph."""
    from deformcontact_b200 import ops, _abi
    sizes = [graph_nodes, 0, 1, graph_nodes // 2 + 3, 64]
    ptr = [0]
    for s_ in sizes:
        ptr.append(ptr[-1] + s_)
    N = ptr[-1]
    gen = torch.Generator().manual_seed(F + graph_nodes)
    eis = []
    for lo, hi in zip(ptr[:-1], ptr[1:]):
        n = hi - lo
        if n == 0:
            continue
        e = torch.randint(0, n, (2, 9 * n), generator=gen)
        e[1, : min(n, 200)] = 0          # one deep row (> 64 edges)
        eis.append(e + lo)
    ei = torch.cat(eis, 1).cuda()
    g = ops.GraphCSR(ei, N, "tag", ptr)
    assert g.tiles_closed and _abi.lib().dc_spmm_stage_supported(g._max_tile, F)
    x = torch.randn(N, F, generator=gen).cuda()
    buf = torch.zeros(N, 3 * F, device="cuda")
    hs = [x] + [buf[:, i * F:(i + 1) * F] for i in range(3)]
    ops.spmm_chain(g.rowptr, g.edges, None, [(hs[i], None, hs[i + 1]) for i in range(3)], tile_ptr=g.tile_ptr, n_tiles=g.n_tiles,
                   max_tile_rows=g._max_tile)
    ref = x
    for i in range(3):
        ref = ops.spmm(g.rowptr, g.nbr, ref, dis=g.dis)
        assert torch.equal(hs[i + 1], ref), f"forward hop {i}"
    adds = [torch.randn(N, F, generator=gen).cuda() for _ in range(3)]
    d = [a.clone() for a in adds]
    g3 = torch.randn(N, F, generator=gen).cuda()
    ops.spmm_chain(g.t[0], g._edges_t, None, [(g3, d[2], d[2]), (d[2], d[1], d[1]), (d[1], d[0], d[0])], tile_ptr=g.tile_ptr,
                   n_tiles=g.n_tiles, max_tile_rows=g._max_tile)
    ref = g3
    for i in (2, 1, 0):
        ref = ops.spmm(g.t[0], g.t[1], ref, dis=g.dis, add=adds[i])
        assert torch.equal(d[i], ref), f"transposed hop {i}"
    # GCN weights (self loop term) through the same kernel
    gg = ops.GraphCSR(ei, N, "gcn", ptr)
    o = torch.empty_like(x)
    ops.spmm_chain(gg.rowptr, gg.edges, gg.self_w, [(x, None, o)], self_loop=True, tile_ptr=gg.tile_ptr, n_tiles=gg.n_tiles,
                   max_tile_rows=gg._max_tile)
    assert torch.equal(o, ops.spmm(gg.rowptr, gg.nbr, x, dis=gg.dis, self_loop=True))


def test_staged_hop_chain_unsupported_tile(dc):
    from deformcontact_b200 import _abi
    assert not _abi.lib().dc_spmm_stage_supported(5000, 256)     # 5000 rows x 64 B do not fit 227 KB
    assert _abi.lib().dc_spmm_stage_supported(3500, 128)


# (307300, 256): the 128-column float4 blocks; (512000, 256) and (195072, 256): the bias gradients of the C3 step
@pytest.mark.parametrize("M,N", [(1, 1), (5000, 256), (2049, 3), (777, 100), (307300, 256), (512000, 256), (195072, 256)])
def test_relu_bwd_colsum_equals_the_two_kernels(dc, M, N):
    """dc_relu_bwd_colsum == dc_relu_bwd followed by dc_colsum, bit for bit (same summation order)."""
    from deformcontact_b200 import ops
    g = torch.Generator().manual_seed(M + N)
    Y = torch.randn(M, N, generator=g).cuda().relu()
    dY = torch.randn(M, N, generator=g).cuda()
    dX, cs = ops.relu_bwd_colsum(Y, dY)
    ref = ops.relu_bwd(Y, dY)
    assert torch.equal(dX, ref) and torch.equal(dX, dY * (Y > 0))
    assert torch.equal(cs, ops.colsum(ref))
    assert_close(cs, ref.double().sum(0).float(), what="colsum")
    # the float4 kernels (N % 4 == 0, aligned rows) and the scalar ones (same data behind a row pitch of N + 1) agree bit for bit
    pad = lambda t: torch.cat([t, torch.zeros(M, 1, device="cuda")], 1)[:, :N]
    dX2, cs2 = ops.relu_bwd_colsum(pad(Y), pad(dY))
    assert torch.equal(dX2, dX) and torch.equal(cs2, cs) and torch.equal(ops.colsum(pad(ref)), cs)


def test_gemm_cta_pairs_on_ragged_shapes(dc):
    """K2 as CTA pairs (cta_group::2): odd numbers of row tiles (the peer CTA's tile lies beyond M), N < 64 (the peer's half of the
    B tile is empty), K not a multiple of 32, every operand layout, single / split-K / batched launches — against fp64."""
    import random
    from deformcontact_b200 import ops
    rnd = random.Random(1)
    g = torch.Generator(device="cuda").manual_seed(1)
    for trial in range(10):
        M = rnd.choice([1, 127, 129, 257, 300, 385, 1000])
        N = rnd.choice([4, 24, 60, 68, 132, 260, 520])
        K = rnd.choice([4, 28, 36, 100, 260, 4100, 20000])
        for ta in (False, True):
            for tb in (False, True):
                Mp, Np, Kp = (M + 3) // 4 * 4, (N + 3) // 4 * 4, (K + 3) // 4 * 4
                A = torch.randn((K, Mp) if ta else (M, Kp), generator=g, device="cuda")[:, :M if ta else K]
                B = torch.randn((N, Kp) if tb else (K, Np), generator=g, device="cuda")[:, :K if tb else N]
                ref = ((A.double().t() if ta else A.double()) @ (B.double().t() if tb else B.double())).float()
                out = ops.gemm([(A, B)], M, N, ta, tb, precision=ops.GEMM_TF32X3)
                assert_close(out, ref, what=f"gemm {M}x{N}x{K} ta={ta} tb={tb}")
                if trial % 3 == 0:
                    outs = [torch.empty(M, N, device="cuda") for _ in range(2)]
                    ops.gemm_batched([(A, B, o) for o in outs], ta, tb)
                    for o in outs:
                        assert_close(o, ref, what=f"gemm_batched {M}x{N}x{K} ta={ta} tb={tb}")
