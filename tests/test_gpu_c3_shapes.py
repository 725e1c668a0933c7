"""The C3 train step that bench.py times, checked at its own size: 256 kNN-8 graphs x 2000 nodes (N = 512 000, E = 4.1 M),
256 colliders x 762 nodes (195 072), hidden 256, 2 attention heads in groups of 4 graphs.

At this size 32-bit offsets, tile and problem tables, split-K part counts and long fp32 chains matter, and the smaller
cases elsewhere in the suite do not reach them:

* K2: every ``ops.gemm`` / ``ops.gemm_batched`` call of one eager step is recorded (shapes, transposes, leading dimensions,
  alignment, epilogue) and each distinct tensor-core signature is replayed on seeded operands against the accuracy contract
  of tests/gemm_contract.py, with the fp64 reference on the GPU, a sentinel-guarded C and a second call giving the same bits;
* K1: the default hop kernels on the C3 kNN structure, bit for bit against the CPU oracle's scatter order;
* the cross attention over 64 groups x 2 heads of 8000 x 3048 and the fused losses at N = 512 000, against fp64;
* the whole step against the fp64 oracle on the GPU: with gradients at 32 graphs (the per-GPU batch of the 8-GPU line),
  forward at 256.
The worst contract values per path are printed at the end (pytest -s)."""
import collections

import pytest
import torch

import oracle
from oracle import convs as oconvs
from gemm_contract import (check_product, epilogue_path, operands, outside_untouched, reference, sentinel_out)
from helpers import (TOL, assert_close, assert_close_arbiter, assert_close_conditioned, gradient_conditioning, rel_err)
from test_gpu_attention import _ref as attention_ref

pytestmark = pytest.mark.gpu

B, NODES, K_NN, GROUP = 256, 2000, 8, 4
RECORD = collections.defaultdict(lambda: [0.0, 0.0])


@pytest.fixture(scope="module")
def dc():
    import deformcontact_b200 as d
    return d


@pytest.fixture(scope="module")
def c3(dc):
    """The batch and model of bench.py's C3 step (bench.py: synthetic.make_batch, seed 0, load_model(attn_group=4))."""
    from deformcontact_b200 import synthetic
    rest, rigid, deformed = synthetic.make_batch(B, NODES, K_NN, first=0, device="cuda")
    torch.manual_seed(0)
    model = dc.load_model(attn_group=GROUP).cuda()
    return model, rest, rigid, deformed


@pytest.fixture(scope="module", autouse=True)
def report():
    yield
    if RECORD:
        print("\nK2 accuracy contract at the C3 step's shapes, worst elementwise / global per path and input class:")
        for (path, cls), (e, g) in sorted(RECORD.items()):
            print(f"  {path:28s} {cls:7s} {e:.2e} {g:.2e}")


def _free():
    torch.cuda.synchronize()
    torch.cuda.empty_cache()


# ----------------------------------------------------------------------------------------------------------------- K2
def _lay(t):
    """(leading dimension, offset in floats from a 16-byte boundary) of a row-major operand."""
    return t.stride(0), (t.data_ptr() % 16) // 4


def _record_calls(dc, monkeypatch, run):
    """Run ``run()`` with ops.gemm / ops.gemm_batched logging every call that reaches dc_gemm / dc_gemm_batched."""
    ops = dc.ops
    gemm, gemm_batched = ops.gemm, ops.gemm_batched
    calls = []

    def rec_gemm(segs, M, N, trans_a=False, trans_b=True, bias=None, relu=False, out=None, accumulate=False,
                 precision=ops.GEMM_AUTO):
        if len(segs) <= dc._abi.MAX_SEGS:   # longer lists are chained by ops.gemm through this function again
            seg = tuple((A.shape[0] if trans_a else A.shape[1]) for A, _ in segs)
            calls.append(("gemm", M, N, seg, bool(trans_a), bool(trans_b), tuple(_lay(A) for A, _ in segs),
                          tuple(_lay(Bm) for _, Bm in segs), _lay(out) if out is not None else (N, 0),
                          None if bias is None else (bias.data_ptr() % 16) // 4, bool(relu), bool(accumulate), int(precision)))
        return gemm(segs, M, N, trans_a=trans_a, trans_b=trans_b, bias=bias, relu=relu, out=out, accumulate=accumulate,
                    precision=precision)

    def rec_batched(problems, trans_a=False, trans_b=True, relu=False, accumulate=False):
        live = [q for q in problems if q[2].numel() > 0]
        tensor = all(_lay(q[0])[0] % 4 == 0 and _lay(q[1])[0] % 4 == 0 and q[0].data_ptr() % 16 == 0 and q[1].data_ptr() % 16 == 0
                     and (q[0].shape[0] if trans_a else q[0].shape[1]) > 0 for q in live)
        if live and tensor:   # otherwise ops.gemm_batched runs one ops.gemm per problem, recorded there
            probs = tuple(((q[0].shape[1] if trans_a else q[0].shape[0]), q[2].shape[1], (q[0].shape[0] if trans_a else q[0].shape[1]),
                           _lay(q[0]), _lay(q[1]), _lay(q[2]), _lay(q[3]) if len(q) > 3 else None) for q in live)
            calls.append(("batched", bool(trans_a), bool(trans_b), bool(relu), bool(accumulate), probs))
        return gemm_batched(problems, trans_a=trans_a, trans_b=trans_b, relu=relu, accumulate=accumulate)

    monkeypatch.setattr(ops, "gemm", rec_gemm)
    monkeypatch.setattr(ops, "gemm_batched", rec_batched)
    try:
        run()
        torch.cuda.synchronize()
    finally:
        monkeypatch.setattr(ops, "gemm", gemm)
        monkeypatch.setattr(ops, "gemm_batched", gemm_batched)
    return calls


def _on_k2(dc, sig):
    """Whether dc_gemm sends a recorded single product to the tensor-core kernel (csrc/gemm.cu: dc_gemm, gemm_tc2_supported)."""
    _, M, N, seg, ta, tb, la, lb, _, _, _, _, prec = sig
    ops = dc.ops
    ok = (all(ld % 4 == 0 and al == 0 for ld, al in la + lb) and (len(seg) == 1 or (not ta and tb)) and M > 0 and N > 0)
    return ok and (prec == ops.GEMM_TF32X3 or prec == ops.GEMM_PREFER_TC or (prec == ops.GEMM_AUTO and M * N * sum(seg) >= 1e8))


def _stored(X, trans, lay, device="cuda"):
    """Logical X stored as the GEMM reads it (X, or with ``trans`` a tensor whose transpose is X) with the recorded
    (leading dimension, 16-byte offset)."""
    Y = X.t() if trans else X
    ld, al = lay
    r, c = Y.shape
    buf = torch.empty(al + max(r - 1, 0) * ld + c, dtype=torch.float32, device=device)
    V = buf.as_strided((r, c), (ld, 1), al)
    V.copy_(Y)
    return V


def _c_out(M, N, lay):
    """A sentinel-guarded C with the recorded row pitch and 16-byte offset."""
    ld, al = lay
    return sentinel_out(M, N, ld, ld + (al - ld) % 4)


def _misaligned(t, al):
    buf = torch.empty(t.numel() + al, dtype=t.dtype, device=t.device)
    v = buf[al:al + t.numel()].view(t.shape)
    v.copy_(t)
    return v


def _replay_gemm(dc, sig, cls, seed):
    _, M, N, seg, ta, tb, la, lb, lc, bias_al, relu, acc, prec = sig
    A, Bm = operands(cls, M, N, sum(seg), seed, device="cuda")
    segs, o = [], 0
    for k, lay_a, lay_b in zip(seg, la, lb):
        segs.append((_stored(A[:, o:o + k], ta, lay_a), _stored(Bm[o:o + k], tb, lay_b)))
        o += k
    del A, Bm
    g = torch.Generator(device="cuda").manual_seed(seed + 1)
    b = None if bias_al is None else _misaligned(torch.randn(N, generator=g, device="cuda"), bias_al)
    c_old = torch.randn(M, N, generator=g, device="cuda") if acc else None
    buf, C = _c_out(M, N, lc)

    def run():
        if acc:
            C.copy_(c_old)
        dc.ops.gemm(segs, M, N, trans_a=ta, trans_b=tb, bias=b, relu=relu, out=C, accumulate=acc, precision=prec)
        return buf.clone()

    first = run()
    what = f"C3 gemm {M}x{N}x{list(seg)} ta={ta} tb={tb} {cls} bias={bias_al} relu={relu} acc={acc}"
    C64, scale = reference(segs, ta, tb, bias=b, c_old=c_old, relu=relu)
    path = ("multi-segment " if len(seg) > 1 else "") + epilogue_path(M, N, sum(-(-k // 32) for k in seg), C, b, acc)
    e, gl = check_product(C, C64, scale, what=what)
    del C64, scale
    outside_untouched(buf, C, what)
    assert torch.equal(first.view(torch.int32), run().view(torch.int32)), f"{what}: second call differs"
    return path, e, gl


def _replay_batched(dc, sig, cls, seed):
    _, ta, tb, relu, acc, probs = sig
    g = torch.Generator(device="cuda").manual_seed(seed + 1)
    qs, bufs, olds = [], [], []
    for j, (M, N, K, la, lb, lc, le) in enumerate(probs):
        A, Bm = operands(cls, M, N, K, seed + 7 * j, device="cuda")
        buf, C = _c_out(M, N, lc)
        q = (_stored(A, ta, la), _stored(Bm, tb, lb), C)
        if le is not None:
            q = q + (_stored(torch.rand(M, N, generator=g, device="cuda"), False, le), torch.randn(M, generator=g, device="cuda"))
        qs.append(q)
        bufs.append(buf)
        olds.append(torch.randn(M, N, generator=g, device="cuda") if acc else None)

    def run():
        for q, c_old in zip(qs, olds):
            if c_old is not None:
                q[2].copy_(c_old)
        dc.ops.gemm_batched(qs, trans_a=ta, trans_b=tb, relu=relu, accumulate=acc)
        return [b.clone() for b in bufs]

    first = run()
    fused = probs[0][6] is not None
    path = "batched " + ("fused " if fused else "") + "K=" + "/".join(str(k) for k in sorted({p[2] for p in probs}))
    worst = [0.0, 0.0]
    for j, (q, c_old, buf) in enumerate(zip(qs, olds, bufs)):
        M, N, K = probs[j][:3]
        what = f"C3 batched problem {j}/{len(probs)} {M}x{N}x{K} ta={ta} tb={tb} {cls} fused={fused} relu={relu} acc={acc}"
        C64, scale = reference([q[:2]], ta, tb, c_old=c_old, E=q[3] if fused else None, rowv=q[4] if fused else None, relu=relu)
        e, gl = check_product(q[2], C64, scale, what=what)
        worst = [max(worst[0], e), max(worst[1], gl)]
        del C64, scale
        outside_untouched(buf, q[2], what)
    assert all(torch.equal(a.view(torch.int32), b.view(torch.int32)) for a, b in zip(first, run())), "C3 batched: second call differs"
    return path, worst[0], worst[1]


def _describe(sig):
    if sig[0] == "gemm":
        _, M, N, seg, ta, tb, la, lb, lc, bias_al, relu, acc, _ = sig
        return (f"gemm M={M} N={N} K={list(seg)} ta={int(ta)} tb={int(tb)} lda={[l for l, _ in la]} ldb={[l for l, _ in lb]} "
                f"ldc={lc[0]} bias={bias_al} relu={int(relu)} acc={int(acc)}")
    _, ta, tb, relu, acc, probs = sig
    shapes = sorted(collections.Counter((M, N, K) for M, N, K, *_ in probs).items())
    return f"batched x{len(probs)} {shapes} ta={int(ta)} tb={int(tb)} fused={probs[0][6] is not None} relu={int(relu)} acc={int(acc)}"


def test_k2_at_the_c3_step_shapes(dc, c3, monkeypatch):
    """Every distinct K2 product of one eager C3 step, replayed on the randn / relu / rowcol classes (plus kblock for
    multi-segment products) against the elementwise and global bounds of the contract; C guarded by sentinels; a second call
    gives the same bits.  All signatures are replayed before the test reports, so a failure lists every failing one."""
    model, rest, rigid, deformed = c3
    model.zero_grad(set_to_none=True)
    calls = _record_calls(dc, monkeypatch, lambda: dc.train_step_loss(model, rest, rigid, deformed)[0].backward())
    model.zero_grad(set_to_none=True)
    _free()
    sigs = list(dict.fromkeys(calls))
    singles = [s for s in sigs if s[0] == "gemm"]
    batched = [s for s in sigs if s[0] == "batched"]
    on_k2 = [s for s in singles if _on_k2(dc, s)]
    print(f"\nC3 step: {len(calls)} GEMM calls, {len(sigs)} distinct signatures; replayed on K2: {len(on_k2)} single + "
          f"{len(batched)} batched; on the exact-fp32 kernel (not K2): {len(singles) - len(on_k2)}")
    # the cases this test exists for: the weight gradients over all nodes, the products over all nodes, the attention batches
    assert any(sum(s[3]) >= B * NODES for s in on_k2), "no K2 product with K >= 512000 recorded"
    assert any(s[1] == B * NODES for s in on_k2), "no K2 product with M = 512000 recorded"
    assert any(len(s[5]) == 2 * B // GROUP and s[5][0][6] is not None for s in batched), "no fused 128-problem batch recorded"
    failed = []
    for i, sig in enumerate(on_k2 + batched):
        multi = sig[0] == "gemm" and len(sig[3]) > 1
        for cls in ("randn", "relu", "rowcol") + (("kblock",) if multi else ()):
            try:
                path, e, gl = (_replay_gemm if sig[0] == "gemm" else _replay_batched)(dc, sig, cls, seed=1000 + 10 * i)
                r = RECORD[(path, cls)]
                r[0], r[1] = max(r[0], e), max(r[1], gl)
            except AssertionError as err:
                failed.append(f"{_describe(sig)} [{cls}]: {str(err).splitlines()[0]}")
            _free()
        print(f"  replayed {_describe(sig)}")
    print(f"C3 K2 signatures failing the contract: {len({f.split(' [')[0] for f in failed})} of {len(on_k2) + len(batched)}")
    assert not failed, "\n".join(failed)


# ----------------------------------------------------------------------------------------------------------------- K1
def _oracle_hop(h, ei, w, n, add=None, bias=None, relu=False):
    """oracle.convs.propagate, starting each receiver's sum at ``add`` (the order K1 uses for a fused addend), then bias, ReLU."""
    if add is None:
        out = oconvs.propagate(h, ei, w, n)
    else:
        msg = w.view(-1, 1) * h.index_select(0, ei[0])
        out = add.clone().scatter_add_(0, ei[1].view(-1, 1).expand_as(msg), msg)
    if bias is not None:
        out = out + bias
    return out.relu() if relu else out


COLS = (slice(0, 32), slice(224, 256))   # hops are column-independent: two 32-column slices keep the CPU oracle small


def _guarded(N, F):
    """A sentinel-guarded [N, F] output: row pitch F + 8, 16-byte aligned, sentinel rows and columns on every side."""
    return sentinel_out(N, F, F + 8, F + 8 + 4)


@pytest.mark.parametrize("variant", ["default", "stream", "stage"])
@pytest.mark.parametrize("mode", ["tag", "gcn"])
def test_k1_at_c3_bit_exact(dc, c3, mode, variant, monkeypatch):
    """The default hop kernels on the C3 kNN structure (tile_ptr from the graph offsets), F = 256: the lean forward and the
    edge-block transposed hop with add / bias / ReLU, the forward chain into slices of a strided [N, 3F] buffer and the
    transposed chain with in-place addends — equal to the CPU oracle (torch.equal) on two column slices, nothing written
    outside the outputs, edge-block status 0.  ``stream`` / ``stage``: the same chains through K1 v11 / v10, bit-identical to
    the default chains."""
    ops = dc.ops
    _, rest, _, _ = c3
    N, F = rest.pos.shape[0], 256
    G = ops.GraphCSR(rest.edge_index, N, mode, rest._ptr_host)
    assert G.tiles_closed and G.n_tiles == B and G._max_tile == NODES
    gen = torch.Generator(device="cuda").manual_seed(3 if mode == "tag" else 4)
    x = torch.randn(N, F, generator=gen, device="cuda")
    adds = [torch.randn(N, F, generator=gen, device="cuda") for _ in range(3)]
    bias = torch.randn(F, generator=gen, device="cuda")

    def chains():
        bufc, hc = _guarded(N, 3 * F)
        hs = [x] + [hc[:, i * F:(i + 1) * F] for i in range(3)]
        ops.propagate_chain(G, [(hs[i], None, hs[i + 1]) for i in range(3)])
        guarded = [_guarded(N, F) for _ in range(3)]
        d = [v for _, v in guarded]
        for di, a in zip(d, adds):
            di.copy_(a)
        ops.propagate_chain(G, [(x, d[2], d[2]), (d[2], d[1], d[1]), (d[1], d[0], d[0])], transpose=True)
        outside_untouched(bufc, hc, "forward chain")
        for i, (bufd, di) in enumerate(guarded):
            outside_untouched(bufd, di, f"transposed chain hop {i}")
        return hs[1:], d

    if variant != "default":
        fwd0, bwd0 = chains()
        fwd0, bwd0 = [t.clone() for t in fwd0], [t.clone() for t in bwd0]
        if variant == "stage":
            assert dc._abi.lib().dc_spmm_stage_supported(G._max_tile, F)
        monkeypatch.setattr(ops, "K1_STREAM" if variant == "stream" else "K1_STAGE", 1)
        fwd, bwd = chains()
        for i in range(3):
            assert torch.equal(fwd[i], fwd0[i]), f"{variant}: forward chain hop {i + 1} differs from the default"
            assert torch.equal(bwd[i], bwd0[i]), f"{variant}: transposed chain hop {i} differs from the default"
        return

    host = lambda t: [t[:, c].cpu() for c in COLS]     # the two column slices, on the host
    outs = {}
    for tr in (False, True):
        for fused in (False, True):
            buf, o = _guarded(N, F)
            G.propagate(x, transpose=tr, add=adds[0] if fused else None, bias=bias if fused else None, relu=fused, out=o)
            outside_untouched(buf, o, f"propagate transpose={tr} fused={fused}")
            outs[(tr, fused)] = host(o)
            del buf, o
    assert int(G.blocks(True).status.item()) == 0, "edge blocks over capacity"
    fwd, bwd = chains()
    fwd, bwd = [host(t) for t in fwd], [host(t) for t in bwd]
    xc, ac, bc = host(x), [host(a) for a in adds], bias.cpu()
    _free()
    ei_n, w = oconvs.gcn_norm(rest.edge_index.cpu(), N, mode == "gcn")
    ei_t = ei_n.flip(0)
    for s, cols in enumerate(COLS):
        h = xc[s]
        for tr, e in ((False, ei_n), (True, ei_t)):
            assert torch.equal(outs[(tr, False)][s], _oracle_hop(h, e, w, N)), f"{mode} propagate transpose={tr} {cols}"
            assert torch.equal(outs[(tr, True)][s], _oracle_hop(h, e, w, N, add=ac[0][s], bias=bc[cols], relu=True)), \
                f"{mode} propagate transpose={tr} add/bias/relu {cols}"
        r = h
        for i in range(3):
            r = _oracle_hop(r, ei_n, w, N)
            assert torch.equal(fwd[i][s], r), f"{mode} forward chain hop {i + 1} {cols}"
        r = h     # the transposed chain starts from x
        for i in (2, 1, 0):
            r = _oracle_hop(r, ei_t, w, N, add=ac[i][s])
            assert torch.equal(bwd[i][s], r), f"{mode} transposed chain hop {i} {cols}"


# ---------------------------------------------------------------------------------------------------- attention, losses
def test_cross_attention_at_c3_grouping(dc, c3):
    """_AttnFn over 64 groups x 2 heads of 8000 x 3048 (F = 256; seeded post-ReLU stand-ins of the encoder outputs), forward
    and backward: out, dxs, dxr, dW, db within 1e-5 of fp64 (the reference formula per group on the GPU), or, where the
    fp32 evaluation of that formula is itself further than that from fp64, as close as it is (fp64 arbiter)."""
    from deformcontact_b200 import attention
    _, rest, rigid, _ = c3
    ps, pr = rest._ptr_host, rigid._ptr_host
    groups = attention._groups(ps, pr, GROUP)
    assert len(groups) == B // GROUP and {(s1 - s0, r1 - r0) for s0, s1, r0, r1 in groups} == {(GROUP * NODES, GROUP * 762)}
    F, H = 256, 2
    g = torch.Generator(device="cuda").manual_seed(5)
    xs = torch.randn(ps[-1], F, generator=g, device="cuda").relu()
    xr = torch.randn(pr[-1], F, generator=g, device="cuda").relu()
    params = []
    for _ in range(H):
        params += [(torch.rand(F, F, generator=g, device="cuda") * 2 - 1) / F ** 0.5 * 0.5,
                   (torch.rand(F, generator=g, device="cuda") * 2 - 1) / F ** 0.5]
    gos = [torch.randn(ps[-1], F, generator=g, device="cuda") for _ in range(H)]

    t = [v.detach().clone().requires_grad_(True) for v in [xs, xr] + params]
    outs = attention._AttnFn.apply(t[0], t[1], groups, *t[2:])
    sum((o * go).sum() for o, go in zip(outs, gos)).backward()
    ours = [o.detach() for o in outs] + [v.grad for v in t]
    del outs, t
    _free()

    def reference(dtype):
        """The reference formula per group (its gradient only reaches the group's rows): outputs and gradients in ``dtype``."""
        p = [v.to(dtype).requires_grad_(True) for v in params]
        res = [torch.zeros(ps[-1], F, dtype=dtype, device="cuda") for _ in range(H)]
        dxs, dxr = torch.zeros_like(xs, dtype=dtype), torch.zeros_like(xr, dtype=dtype)
        for s0, s1, r0, r1 in groups:
            a = xs[s0:s1].to(dtype).requires_grad_(True)
            b = xr[r0:r1].to(dtype).requires_grad_(True)
            loss = 0.0
            for h in range(H):
                o = attention_ref(a, b, p[2 * h], p[2 * h + 1], [(0, s1 - s0, 0, r1 - r0)])
                res[h][s0:s1] = o.detach()
                loss = loss + (o * gos[h][s0:s1].to(dtype)).sum()
            loss.backward()
            dxs[s0:s1], dxr[r0:r1] = a.grad, b.grad
        return res + [dxs, dxr] + [v.grad for v in p]

    r64 = reference(torch.float64)
    r32 = reference(torch.float32)
    names = [f"out{h}" for h in range(H)] + ["dxs", "dxr"] + [f"{n}{h}" for h in range(H) for n in ("dW", "db")]
    for name, a, b32, b64 in zip(names, ours, r32, r64):
        e = rel_err(a, b64)
        if e > TOL:
            assert_close_arbiter(a, b32, b64, what=f"C3 attention {name}")
        print(f"C3 attention {name}: {e:.2e} from fp64 (fp32 formula {rel_err(b32, b64):.2e})")
    del r64, r32
    _free()


def test_edge_loss_at_c3_size_vs_fp64(dc, c3):
    """dc_edge_loss (L1 + gradient consistency and their gradients) on the C3 soft graph, N = 512 000, E = 4.1 M, against
    F.l1_loss + GradientConsistencyLoss evaluated in fp64 on the GPU."""
    _, rest, _, _ = c3
    N = rest.pos.shape[0]
    g = torch.Generator(device="cuda").manual_seed(7)
    pred = torch.randn(N, 3, generator=g, device="cuda") * 0.01
    tgt = torch.randn(N, 3, generator=g, device="cuda") * 0.01
    p = pred.clone().requires_grad_(True)
    l1, lc = dc.fused_losses(dc.Data(x=p, edge_index=rest.edge_index, pos=p), dc.Data(x=tgt, edge_index=rest.edge_index, pos=tgt))
    (0.7 * l1 + 1.3 * lc).backward()
    p64 = pred.double().requires_grad_(True)
    t64 = tgt.double()
    r1 = torch.nn.functional.l1_loss(p64, t64)
    rc = oracle.GradientConsistencyLoss()(oracle.Data(x=p64, edge_index=rest.edge_index, pos=p64),
                                          oracle.Data(x=t64, edge_index=rest.edge_index, pos=t64))
    (0.7 * r1 + 1.3 * rc).backward()
    for name, a, b in (("l1", l1, r1), ("consistency", lc, rc), ("dpred", p.grad, p64.grad)):
        assert_close(a, b.detach(), what=f"C3 edge loss {name} vs fp64")


# ------------------------------------------------------------------------------------------------------- whole step
def _to64(b):
    out = oracle.Batch(x=b.x.double(), edge_index=b.edge_index, pos=b.pos.double())
    out.ptr, out.batch = b.ptr, b.batch
    return out


def _oracle_model(model, dtype):
    ref = oracle.load_model(attn_group=GROUP).to(device="cuda", dtype=dtype)
    ref.load_state_dict(model.state_dict())
    return ref


def test_whole_step_32_graphs_vs_fp64_oracle(dc, c3):
    """The per-GPU batch of the 8-GPU line (32 graphs, 64 000 nodes): losses and the predicted displacement within 1e-5 of
    the fp64 oracle on the GPU; every parameter gradient within 1e-5 of the fp32 oracle on the GPU, or the fp64 arbiter, or
    the movement of the fp64 gradients under a 1e-6 relative perturbation of the weights (the C1 test's bar)."""
    model, _, _, _ = c3
    n = 32
    from deformcontact_b200 import synthetic
    rest, rigid, deformed = synthetic.make_batch(n, NODES, K_NN, first=0, device="cuda")
    model.zero_grad(set_to_none=True)
    loss_o, l1_o, lc_o = dc.train_step_loss(model, rest, rigid, deformed)
    loss_o.backward()
    with torch.no_grad():
        disp_o = model(rest, rigid).pos - rest.pos
    ref32, ref64 = _oracle_model(model, torch.float32), _oracle_model(model, torch.float64)
    oracle.train_step_loss(ref32, rest, rigid, deformed)[0].backward()
    r64, g64, d64 = _to64(rest), _to64(rigid), _to64(deformed)
    loss_64, l1_64, lc_64 = oracle.train_step_loss(ref64, r64, g64, d64)
    loss_64.backward()
    with torch.no_grad():
        disp_64 = ref64(r64, g64).pos - r64.pos
    for name, a, b in (("loss", loss_o, loss_64), ("L1 loss", l1_o, l1_64), ("consistency loss", lc_o, lc_64),
                       ("predicted displacement", disp_o, disp_64)):
        assert_close(a, b.detach(), what=f"32 graphs {name} vs fp64")
    cond = gradient_conditioning(ref64, lambda m: oracle.train_step_loss(m, r64, g64, d64)[0], eps=1e-6, samples=3)
    worst, widened = 0.0, []
    for (k, po), (_, pr), (_, p64) in zip(model.named_parameters(), ref32.named_parameters(), ref64.named_parameters()):
        assert po.grad is not None, k
        e = assert_close_conditioned(po.grad, pr.grad, p64.grad, cond[k], what=f"32 graphs d{k}")
        worst = max(worst, e)
        if e > max(TOL, 2.0 * rel_err(pr.grad, p64.grad)):
            widened.append((k, e, cond[k]))
    model.zero_grad(set_to_none=True)
    print(f"\n32-graph step: worst gradient error {worst:.2e}; parameters judged by the perturbation bound: {widened}; "
          f"peak device memory {torch.cuda.max_memory_allocated() / 2 ** 30:.1f} GiB")
    del ref32, ref64, cond
    _free()


def test_whole_step_256_graphs_forward_vs_fp64_oracle(dc, c3):
    """The C3 step itself: losses and the predicted displacement within 1e-5 of the fp64 oracle's forward on the GPU (no
    gradients here: they are checked at 32 graphs above; the peak memory of this forward is printed)."""
    model, rest, rigid, deformed = c3
    with torch.no_grad():
        loss_o, l1_o, lc_o = dc.train_step_loss(model, rest, rigid, deformed)
        disp_o = model(rest, rigid).pos - rest.pos
        ref64 = _oracle_model(model, torch.float64)
        r64, g64, d64 = _to64(rest), _to64(rigid), _to64(deformed)
        torch.cuda.reset_peak_memory_stats()
        loss_64, l1_64, lc_64 = oracle.train_step_loss(ref64, r64, g64, d64)
        disp_64 = ref64(r64, g64).pos - r64.pos
        peak = torch.cuda.max_memory_allocated()
    for name, a, b in (("loss", loss_o, loss_64), ("L1 loss", l1_o, l1_64), ("consistency loss", lc_o, lc_64),
                       ("predicted displacement", disp_o, disp_64)):
        e = assert_close(a, b, what=f"C3 {name} vs fp64")
        print(f"C3 {name}: {e:.2e} from fp64")
    print(f"C3 fp64 oracle forward: peak device memory {peak / 2 ** 30:.1f} GiB")
    del ref64, r64, g64, d64, disp_64
    _free()
