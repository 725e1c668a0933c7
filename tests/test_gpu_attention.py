"""N1: the dense cross attention (models/model.py:7-21) on libdcb200 — forward and hand-derived backward against
the reference formula in fp32 and, where the unscaled softmax makes fp32 itself ill-conditioned, the fp64 arbiter."""
import pytest
import torch

from helpers import assert_close, assert_close_arbiter

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def dc():
    import deformcontact_b200 as d
    return d


def _ref(xs, xr, W, b, groups):
    """models/model.py:14-19 applied per attention group."""
    outs = []
    for s0, s1, r0, r1 in groups:
        q, k = xs[s0:s1] @ W.T + b, xr[r0:r1] @ W.T + b
        outs.append(torch.softmax(q @ k.T, dim=-1) @ xr[r0:r1])
    return torch.cat(outs, 0)


@pytest.mark.parametrize("F,ptr_s,ptr_r,group", [
    (64, [0, 300, 700, 1000, 1500], [0, 40, 100, 180, 240], 2),       # ragged groups
    (256, [0, 2000, 4000], [0, 764, 1528], None),                      # whole batch, N-chunked scores (1528 > 256)
    (32, [0, 130, 131, 400], [0, 36, 40, 72], 1),                      # tiny groups (SIMT fallback below the size cut)
    (128, [0, 1000, 2000], [0, 381, 763], 1),                          # nr % 4 != 0 in one group (fallback layout path)
])
def test_cross_attention_forward_backward(dc, F, ptr_s, ptr_r, group):
    from deformcontact_b200 import attention
    g = torch.Generator().manual_seed(F)
    Ns, Nr = ptr_s[-1], ptr_r[-1]
    xs = torch.randn(Ns, F, generator=g).relu()            # encoder outputs are post-ReLU
    xr = torch.randn(Nr, F, generator=g).relu()
    W = (torch.rand(F, F, generator=g) * 2 - 1) / F ** 0.5 * 0.5
    b = (torch.rand(F, generator=g) * 2 - 1) / F ** 0.5
    go = torch.randn(Ns, F, generator=g)
    groups = attention._groups(ptr_s, ptr_r, group)

    def run(dtype, dev):
        t = [v.detach().clone().to(dtype=dtype, device=dev).requires_grad_(True) for v in (xs, xr, W, b)]
        if dev == "cuda":
            out = attention._AttnFn.apply(t[0], t[1], groups, t[2], t[3])[0]
        else:
            out = _ref(*t, groups)
        out.backward(go.to(dtype=dtype, device=dev))
        return [out] + [v.grad for v in t]

    ours, r32, r64 = run(torch.float32, "cuda"), run(torch.float32, "cpu"), run(torch.float64, "cpu")
    for name, a, b32, b64 in zip(("out", "dxs", "dxr", "dW", "db"), ours, r32, r64):
        assert_close_arbiter(a, b32, b64, what=f"attention {name} F={F}")


def test_softmax_rows_kernels(dc):
    from deformcontact_b200 import attention
    g = torch.Generator().manual_seed(0)
    for M, N in [(37, 1), (64, 3048), (5, 5000), (300, 257)]:
        S = (torch.randn(M, N, generator=g) * 8).cuda()
        ref = torch.softmax(S.double(), -1)
        P = attention.softmax_rows_(S.clone())
        assert_close(P, ref.float(), what=f"softmax {M}x{N}")
        dP = torch.randn(M, N, generator=g).cuda()
        ref_d = ref * (dP.double() - (dP.double() * ref).sum(-1, keepdim=True))
        dS = attention.softmax_bwd_rows_(ref.float().contiguous(), dP.clone())
        assert_close(dS, ref_d.float(), tol=2e-5, what=f"softmax bwd {M}x{N}")
        # strided views (padded rows)
        buf = torch.zeros(M, N + 3).cuda()
        buf[:, :N] = S
        assert torch.equal(attention.softmax_rows_(buf[:, :N]), P)


def test_gemm_tc_wide_n_and_ragged_k(dc):
    """K2 with N > 256 (column chunks) and K % 32 != 0 (TMA zero fill) against fp64."""
    from deformcontact_b200 import ops
    g = torch.Generator().manual_seed(1)
    for M, N, K, tb in [(1000, 3048, 256, True), (777, 600, 3048, False), (300, 257 * 4, 100, True), (2000, 256, 3048, False)]:
        A = torch.randn(M, K, generator=g).cuda()
        B = (torch.randn(N, K, generator=g) if tb else torch.randn(K, N, generator=g)).cuda()
        ref = A.double() @ (B.double().T if tb else B.double())
        out = ops.gemm([(A, B)], M, N, trans_b=tb, precision=dc._abi.GEMM_TF32X3)
        assert_close(out, ref.float(), what=f"gemm_tc {M}x{N}x{K}")
        out2 = ops.gemm([(A, B)], M, N, trans_b=tb, precision=dc._abi.GEMM_FP32)
        assert_close(out2, ref.float(), what=f"gemm_simt {M}x{N}x{K}")


@pytest.mark.parametrize("widths,N,relu", [((256, 256, 256), 256, True), ((64,), 3, False), ((32, 96), 40, True), ((21,), 16, False)])
def test_mlp_linear_segments(dc, widths, N, relu):
    """mlp.linear == act(cat(segs) @ W.T + b), forward and backward, without the concatenation."""
    from deformcontact_b200 import mlp
    g = torch.Generator().manual_seed(N)
    M = 1500
    segs = [torch.randn(M, w, generator=g) for w in widths]
    W = torch.randn(N, sum(widths), generator=g) / sum(widths) ** 0.5
    b = torch.randn(N, generator=g)
    go = torch.randn(M, N, generator=g)

    def run(dtype, dev):
        t = [v.detach().clone().to(dtype=dtype, device=dev).requires_grad_(True) for v in [W, b] + segs]
        if dev == "cuda":
            y = mlp.linear(t[2:], t[0], t[1], relu)
        else:
            y = torch.cat(t[2:], 1) @ t[0].T + t[1]
            y = y.relu() if relu else y
        y.backward(go.to(dtype=dtype, device=dev))
        return [y] + [v.grad for v in t]

    ours, r32, r64 = run(torch.float32, "cuda"), run(torch.float32, "cpu"), run(torch.float64, "cpu")
    for i, (a, b32, b64) in enumerate(zip(ours, r32, r64)):
        assert_close_arbiter(a, b32, b64, what=f"linear tensor {i}")


def test_gemm_batched(dc):
    """dc_gemm_batched == per-problem dc_gemm (same kernel, same chain structure => bit-identical), every layout,
    ragged sizes, empty problems, and the fallback when a problem does not fit the tensor path."""
    from deformcontact_b200 import ops
    g = torch.Generator().manual_seed(3)
    shapes = [(300, 520, 256), (1, 17, 40), (129, 128, 3048), (1000, 256, 36), (0, 64, 64), (257, 64, 8)]
    for ta in (False, True):
        for tb in (False, True):
            probs, refs = [], []
            for M, N, K in shapes:
                A = torch.randn((K, (M + 3) // 4 * 4) if ta else (M, K), generator=g).cuda()
                if ta:
                    A = A[:, :M]
                B = (torch.randn(N, K, generator=g) if tb else torch.randn(K, (N + 3) // 4 * 4, generator=g)).cuda()
                if not tb:
                    B = B[:, :N]
                Cm = torch.zeros(M, N).cuda()
                probs.append((A, B, Cm))
                refs.append(ops.gemm([(A, B)], M, N, trans_a=ta, trans_b=tb, precision=dc._abi.GEMM_TF32X3) if M else Cm.clone())
            ops.gemm_batched(probs, trans_a=ta, trans_b=tb)
            for (A, B, Cm), ref, (M, N, K) in zip(probs, refs, shapes):
                if M == 129 and K == 3048:
                    # the single-problem launch splits K into parts (different summation tree): compare against fp64
                    r64 = (A.double().T if ta else A.double()) @ (B.double().T if tb else B.double())
                    assert_close(Cm, r64.float(), what="batched vs fp64")
                else:
                    assert torch.equal(Cm, ref), (ta, tb, M, N, K)
    # a problem with an unaligned leading dimension sends the whole batch down the per-problem path
    A = torch.randn(64, 21, generator=g).cuda(); B = torch.randn(32, 21, generator=g).cuda(); Cm = torch.empty(64, 32).cuda()
    ops.gemm_batched([(A, B, Cm)], trans_b=True)
    assert_close(Cm, (A.double() @ B.double().T).float(), what="fallback")


def test_gemm_batched_fused_epilogue(dc):
    """C = E o (A B^T - rowv[:, None]) (the fused softmax backward) and dc_rowdot."""
    from deformcontact_b200 import ops
    g = torch.Generator().manual_seed(4)
    probs, refs = [], []
    for M, N, K in [(300, 520, 64), (129, 36, 256), (1000, 3048, 32)]:
        A, B = torch.randn(M, K, generator=g).cuda(), torch.randn(N, K, generator=g).cuda()
        E = torch.rand((M, (N + 3) // 4 * 4), generator=g).cuda()[:, :N]
        rv = torch.randn(M, generator=g).cuda()
        Cm = torch.empty(M, N).cuda()
        probs.append((A, B, Cm, E, rv))
        refs.append(E.double() * (A.double() @ B.double().T - rv.double()[:, None]))
    ops.gemm_batched(probs, trans_b=True)
    for (A, B, Cm, E, rv), ref in zip(probs, refs):
        assert_close(Cm, ref.float(), what="fused epilogue")
    X, Y = torch.randn(777, 100, generator=g).cuda(), torch.randn(777, 100, generator=g).cuda()
    assert_close(ops.rowdot(X, Y), (X.double() * Y.double()).sum(1).float(), what="rowdot")


def test_fused_losses(dc):
    """N2: dc_edge_loss == (F.l1_loss, GradientConsistencyLoss) of train.py:47-58, values and gradients (fp64 arbiter);
    duplicate edges, self loops (zero-length edge vectors), isolated nodes."""
    import oracle
    g = torch.Generator().manual_seed(7)
    N = 1500
    ei = torch.randint(0, N - 50, (2, 9000), generator=g)
    ei = torch.cat([ei, torch.arange(20).repeat(2, 1), ei[:, :100]], 1)      # self loops + duplicates
    pred_pos = torch.randn(N, 3, generator=g) * 0.01
    tgt_pos = torch.randn(N, 3, generator=g) * 0.01
    pred_pos[5] = tgt_pos[5]                                                  # exact zeros in the L1 term

    def run(dtype, dev, fused):
        p = pred_pos.detach().clone().to(dtype=dtype, device=dev).requires_grad_(True)
        t = tgt_pos.to(dtype=dtype, device=dev)
        if fused:
            a = dc.Data(x=p, edge_index=ei.to(dev), pos=p)
            b = dc.Data(x=t, edge_index=ei.to(dev), pos=t)
            l1, lc = dc.fused_losses(a, b)
        else:
            a = oracle.Data(x=p, edge_index=ei, pos=p)
            b = oracle.Data(x=t, edge_index=ei, pos=t)
            l1, lc = torch.nn.functional.l1_loss(p, t), oracle.GradientConsistencyLoss()(a, b)
        (0.7 * l1 + 1.3 * lc).backward()
        return [l1.detach(), lc.detach(), p.grad]

    ours, r32, r64 = run(torch.float32, "cuda", True), run(torch.float32, "cpu", False), run(torch.float64, "cpu", False)
    for name, a, b32, b64 in zip(("l1", "consistency", "dpred"), ours, r32, r64):
        assert_close_arbiter(a, b32, b64, what=f"fused loss {name}")
    again = run(torch.float32, "cuda", True)
    assert all(torch.equal(x, y) for x, y in zip(ours, again)), "deterministic"


def test_gemm_tma_epilogue_equals_the_staged_epilogue_bit_for_bit(dc):
    """K2 TMA epilogue (gemm_tc2.cu, template TEPI: contractions K <= 512 of CTA pairs without accumulate) against the staged
    epilogue on the same products, in process: (a) a batch of short-K problems runs with TMA epilogues; the same problems
    followed by ONE long-K problem send the whole launch down the staged path; (b) a single product with bias + ReLU against
    the same product accumulated onto zeros (accumulate disables the TMA epilogue).  Ragged M / N (clipped TMA boxes), odd row
    tile counts (the pair's missing tile), every layout, plain and fused (C = E o (acc - rowv)) epilogues."""
    from deformcontact_b200 import ops
    g = torch.Generator(device="cuda").manual_seed(9)
    rn = lambda *s: torch.randn(*s, generator=g, device="cuda")
    shapes = [(300, 520, 256), (129, 36, 64), (1000, 3048, 32), (31, 4, 512), (257, 100, 96)]
    for ta in (False, True):
        for tb in (False, True):
            for fused in (False, True):
                if fused and (ta or not tb):
                    continue
                def build():
                    probs = []
                    gg = torch.Generator(device="cuda").manual_seed(10)
                    for M, N, K in shapes:
                        Mp, Np = (M + 3) // 4 * 4, (N + 3) // 4 * 4
                        A = torch.randn((K, Mp) if ta else (M, K), generator=gg, device="cuda")[:, :M if ta else K]
                        B = torch.randn((N, K) if tb else (K, Np), generator=gg, device="cuda")[:, :K if tb else N]
                        Cm = torch.full((M, Np), -7.0, device="cuda")[:, :N]          # row pitch % 4 == 0 (TMA), N itself ragged
                        if fused:
                            E = torch.rand((M, Np), generator=gg, device="cuda")[:, :N]
                            probs.append((A, B, Cm, E, torch.randn(M, generator=gg, device="cuda")))
                        else:
                            probs.append((A, B, Cm))
                    return probs
                tma = build()
                ops.gemm_batched(tma, trans_a=ta, trans_b=tb)
                staged = build()
                Kl = 1024
                Al = rn(Kl, 64) if ta else rn(64, Kl)
                Bl = rn(64, Kl) if tb else rn(Kl, 64)
                long_problem = (Al, Bl, torch.empty(64, 64, device="cuda")) + ((torch.rand(64, 64, device="cuda"), rn(64)) if fused else ())
                ops.gemm_batched(staged + [long_problem], trans_a=ta, trans_b=tb)
                for i, (p, q) in enumerate(zip(tma, staged)):
                    assert torch.equal(p[2], q[2]), (ta, tb, fused, shapes[i])
                    if fused:
                        ref = p[3].double() * ((p[0].double() @ p[1].double().T) - p[4].double()[:, None])
                        assert_close(p[2], ref.float(), what=f"fused TMA epilogue {shapes[i]}")
    for M, N, K in [(300, 520, 256), (129, 36, 64), (4000, 256, 256)]:
        A, B, b = rn(M, K), rn(N, K), rn(N)
        for relu in (False, True):
            out_tma = ops.gemm([(A, B)], M, N, bias=b, relu=relu, precision=dc._abi.GEMM_TF32X3)
            out_staged = ops.gemm([(A, B)], M, N, bias=b, relu=relu, out=torch.zeros(M, N, device="cuda"), accumulate=True,
                                  precision=dc._abi.GEMM_TF32X3)
            assert torch.equal(out_tma, out_staged), (M, N, K, relu)
            ref = A.double() @ B.double().T + b.double()
            assert_close(out_tma, (ref.relu() if relu else ref).float(), what="TMA epilogue bias / relu")


@pytest.mark.parametrize("case", ["three_heads", "empty_groups", "peaked"])
def test_cross_attention_heads_empty_groups_peaked(dc, case):
    """_AttnFn over H = 3 heads (one batched launch per product type over heads x groups; dxs and dxr summed over heads),
    a group without resting nodes next to a group without collider nodes (the zero fills of rows no live group writes), and
    a peaked softmax (row max P >= 0.9 on most rows), where the unscaled softmax amplifies score error."""
    from deformcontact_b200 import attention
    H, ptr_s, ptr_r, wscale = {
        "three_heads": (3, [0, 300, 700, 1000], [0, 40, 100, 180], 0.5),
        "empty_groups": (2, [0, 300, 300, 700, 1000], [0, 40, 90, 90, 150], 0.5),
        "peaked": (1, [0, 500, 1000], [0, 200, 400], 6.0),
    }[case]
    F = 64
    g = torch.Generator().manual_seed(11)
    Ns, Nr = ptr_s[-1], ptr_r[-1]
    xs = torch.randn(Ns, F, generator=g).relu()
    xr = torch.randn(Nr, F, generator=g).relu()
    params = []
    for _ in range(H):
        params += [(torch.rand(F, F, generator=g) * 2 - 1) / F ** 0.5 * wscale, (torch.rand(F, generator=g) * 2 - 1) / F ** 0.5]
    gos = [torch.randn(Ns, F, generator=g) for _ in range(H)]
    groups = attention._groups(ptr_s, ptr_r, 1)
    if case == "peaked":
        W, b = params
        pmax = torch.cat([torch.softmax((xs[s0:s1] @ W.T + b) @ (xr[r0:r1] @ W.T + b).T, -1).max(-1).values
                          for s0, s1, r0, r1 in groups])
        assert (pmax >= 0.9).float().mean() >= 0.8

    def run(dtype, dev):
        t = [v.detach().clone().to(dtype=dtype, device=dev).requires_grad_(True) for v in [xs, xr] + params]
        if dev == "cuda":
            outs = attention._AttnFn.apply(t[0], t[1], groups, *t[2:])
        else:
            outs = [_ref(t[0], t[1], t[2 + 2 * h], t[3 + 2 * h], groups) for h in range(H)]
        sum((o * go.to(dtype=dtype, device=dev)).sum() for o, go in zip(outs, gos)).backward()
        return list(outs) + [v.grad for v in t]

    ours, r32, r64 = run(torch.float32, "cuda"), run(torch.float32, "cpu"), run(torch.float64, "cpu")
    names = [f"out{h}" for h in range(H)] + ["dxs", "dxr"] + [f"{n}{h}" for h in range(H) for n in ("dW", "db")]
    for name, a, b32, b64 in zip(names, ours, r32, r64):
        assert_close_arbiter(a, b32, b64, what=f"attention {case} {name}")
