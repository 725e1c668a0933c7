"""Every path of the tensor-core GEMM (K2, csrc/gemm_tc2.cu) against the accuracy contract of tests/gemm_contract.py.

A pairwise covering set over layouts, shapes (odd row-tile counts leave a CTA pair's second tile empty; N < 64 leaves the
peer's half of B empty; K from 4 to 70001), split-K, epilogues (TMA, staged, scalar stores,
bias aligned and not), multi-segment products with ragged segment widths (TMA zero fill per segment, k parts that end inside
a segment, more than four segments chained), batched products (mixed sizes, empty problems, the fused epilogue) and the
AUTO dispatch.  Every product also checks that nothing outside C changed (C is a view into a buffer filled with a sentinel
bit pattern) and that a second call gives the same bits.  The worst values per path and input class are printed at the end
(pytest -s)."""
import collections

import pytest
import torch

from gemm_contract import CLASSES, check_product, epilogue_path, operands, outside_untouched, reference, sentinel_out, stored

pytestmark = pytest.mark.gpu

RECORD = collections.defaultdict(lambda: [0.0, 0.0])


@pytest.fixture(scope="module")
def dc():
    import deformcontact_b200 as d
    return d


@pytest.fixture(scope="module", autouse=True)
def report():
    yield
    if RECORD:
        print("\nK2 accuracy contract, worst elementwise / global per path and input class:")
        for (path, cls), (e, g) in sorted(RECORD.items()):
            print(f"  {path:28s} {cls:7s} {e:.2e} {g:.2e}")


def _record(path, cls, C, C64, scale, what):
    e, g = check_product(C, C64, scale, what=what)
    r = RECORD[(path, cls)]
    r[0], r[1] = max(r[0], e), max(r[1], g)


def _out(M, N, layout):
    """A sentinel-filled buffer and the C view into it: 'aligned' (16-byte aligned, ldc % 4 == 0), 'ldc' (ldc % 4 == 1) or
    'offset' (C one float past a 16-byte boundary)."""
    Np = (N + 3) // 4 * 4
    width, c0 = {"aligned": (Np + 8, 4), "ldc": (Np + 9, 4), "offset": (Np + 8, 1)}[layout]
    return sentinel_out(M, N, width, width + c0)


def _bias(N, kind, g):
    if kind is None:
        return None
    b = torch.randn(N + 1, generator=g, device="cuda")
    return b[:N] if kind == "aligned" else b[1:]


def _single(dc, M, N, Ks, ta, tb, cls, bias=None, relu=False, accumulate=False, out="aligned", precision=None, seed=0):
    ops = dc.ops
    precision = ops.GEMM_TF32X3 if precision is None else precision
    Ktot = sum(Ks)
    A, B = operands(cls, M, N, Ktot, seed, device="cuda")
    if len(Ks) == 1:
        segs = [(stored(A, ta), stored(B, tb))]
    else:   # column blocks of one K-major pair, as the decoder and TAGConv layer inputs are laid out
        As, Bs = stored(A, False), stored(B, True)
        offs = [sum(Ks[:i]) for i in range(len(Ks))]
        segs = [(As[:, o:o + k], Bs[:, o:o + k]) for o, k in zip(offs, Ks)]
    g = torch.Generator(device="cuda").manual_seed(seed + 1)
    b = _bias(N, bias, g)
    c_old = torch.randn(M, N, generator=g, device="cuda") if accumulate else None
    buf, C = _out(M, N, out)
    what = f"{M}x{N}x{list(Ks)} ta={ta} tb={tb} {cls} bias={bias} relu={relu} acc={accumulate} out={out}"

    def run():
        if accumulate:
            C.copy_(c_old)
        ops.gemm(segs, M, N, trans_a=ta, trans_b=tb, bias=b, relu=relu, out=C, accumulate=accumulate, precision=precision)
        return buf.clone()

    first = run()
    C64, scale = reference(segs, ta, tb, bias=b, c_old=c_old, relu=relu)
    kbs = [-(-k // 32) for k in Ks]
    path = "multi-segment " if len(Ks) > 1 else ""
    path += "chained" if len(Ks) > 4 else epilogue_path(M, N, sum(kbs), C, b, accumulate)
    _record(path, cls, C, C64, scale, what)
    outside_untouched(buf, C, what)
    assert torch.equal(first.view(torch.int32), run().view(torch.int32)), f"{what}: second call differs"
    return C.clone()


# (M, N, K, ta, tb, epilogue): a pairwise covering set of shapes x layouts x epilogues
SINGLE = [
    (1, 4, 4, 0, 1, {}),
    (127, 60, 36, 1, 0, dict(bias="aligned")),
    (129, 129, 100, 0, 0, dict(bias="misaligned", relu=True)),
    (257, 520, 512, 1, 1, dict(bias="aligned", relu=True)),
    (1000, 4, 544, 0, 1, dict(accumulate=True)),
    (1, 60, 4100, 1, 1, dict(out="ldc")),
    (127, 129, 70001, 0, 1, dict(bias="misaligned", relu=True, accumulate=True)),
    (129, 520, 4, 1, 0, dict(out="offset")),
    (257, 4, 36, 0, 0, dict(bias="misaligned")),
    (1000, 60, 100, 1, 1, dict(out="ldc", relu=True)),
    (1, 129, 512, 0, 0, dict(bias="aligned")),
    (127, 520, 544, 1, 0, dict(out="offset", accumulate=True)),
    (129, 4, 4100, 0, 1, dict(relu=True)),
    (257, 60, 70001, 1, 0, dict(bias="aligned")),
    (1000, 129, 36, 0, 1, dict(out="offset", relu=True)),
    (1000, 520, 100, 1, 0, dict(bias="misaligned")),
    (257, 129, 4, 1, 1, dict(accumulate=True, bias="aligned")),
    (127, 4, 100, 1, 1, dict(out="ldc", bias="misaligned")),
    (129, 60, 544, 0, 0, dict(bias="misaligned", relu=True)),
    (1, 520, 36, 1, 0, dict(out="ldc", accumulate=True)),
    (1000, 520, 4100, 0, 0, dict(out="offset", bias="aligned")),
    (257, 129, 70001, 1, 1, dict(out="ldc")),
]


@pytest.mark.parametrize("M,N,K,ta,tb,epi", SINGLE)
def test_single_product(dc, M, N, K, ta, tb, epi):
    i = SINGLE.index((M, N, K, ta, tb, epi))
    _single(dc, M, N, (K,), bool(ta), bool(tb), CLASSES[i % len(CLASSES)], seed=i, **epi)


# one shape per epilogue path, every input class: TMA epilogue, staged (accumulate), scalar stores, split-K with bias and
# ReLU, and a long contraction with random signs; the layouts rotate with the class
CLASS_SHAPES = [
    (257, 128, 256, dict(bias="aligned")),
    (129, 520, 100, dict(accumulate=True)),
    (1000, 60, 36, dict(out="offset", bias="misaligned", relu=True)),
    (127, 129, 4100, dict(bias="misaligned", relu=True)),
    (129, 60, 70001, dict(accumulate=True)),
]


@pytest.mark.parametrize("cls", CLASSES)
@pytest.mark.parametrize("shape", range(len(CLASS_SHAPES)))
def test_input_classes(dc, cls, shape):
    M, N, K, epi = CLASS_SHAPES[shape]
    i = CLASSES.index(cls) + shape
    _single(dc, M, N, (K,), bool(i & 1), bool(i & 2), cls, seed=100 + 10 * shape + CLASSES.index(cls), **epi)


MULTI = [
    ((36, 100), 257, 60, dict(bias="aligned")),                          # one part, TMA epilogue
    ((100, 28, 260), 129, 520, dict(bias="misaligned")),                  # ragged widths, one part
    ((260, 100, 28, 260), 1000, 129, dict(relu=True, accumulate=True)),    # 2 parts: the boundary at k-block 16 is inside segment 4
    ((260, 260, 36), 127, 4, dict(out="ldc", bias="aligned")),            # 2 parts: the boundary at k-block 16 is inside segment 2
    ((100, 28, 260, 36, 100, 28), 257, 520, dict(bias="aligned", relu=True)),   # > 4 segments: chained with accumulate
    ((28, 36, 100, 260, 36), 129, 60, dict(out="offset")),
]


@pytest.mark.parametrize("cls", ["randn", "kblock", "rowcol", "relu"])
@pytest.mark.parametrize("case", range(len(MULTI)))
def test_multi_segment(dc, case, cls):
    Ks, M, N, epi = MULTI[case]
    _single(dc, M, N, Ks, False, True, cls, seed=200 + case, **epi)


def _batched(dc, shapes, ta, tb, cls, relu=False, accumulate=False, fused=False, out="aligned", lde_pad=0, seed=0):
    """shapes: [(M, N, K)]; fused: every problem carries E (rows padded by lde_pad floats beyond a multiple of 4) and rowv."""
    ops = dc.ops
    g = torch.Generator(device="cuda").manual_seed(seed + 1)
    probs, refs, bufs = [], [], []
    for j, (M, N, K) in enumerate(shapes):
        A, B = operands(cls, M, N, K, seed + 7 * j, device="cuda")
        A, B = stored(A, ta), stored(B, tb)
        buf, C = _out(M, N, out)
        c_old = torch.randn(M, N, generator=g, device="cuda") if accumulate else None
        q = (A, B, C)
        if fused:
            ld = (N + 3) // 4 * 4 + lde_pad
            E = torch.rand((M, ld), generator=g, device="cuda")[:, :N]
            q = q + (E, torch.randn(M, generator=g, device="cuda"))
        probs.append(q)
        bufs.append((buf, c_old))
        refs.append(reference([(A, B)], ta, tb, c_old=c_old, E=q[3] if fused else None, rowv=q[4] if fused else None, relu=relu))

    def run():
        for (buf, c_old), q in zip(bufs, probs):
            if c_old is not None:
                q[2].copy_(c_old)
        ops.gemm_batched(probs, trans_a=ta, trans_b=tb, relu=relu, accumulate=accumulate)
        return [buf.clone() for buf, _ in bufs]

    first = run()
    if fused:
        tma = out == "aligned" and lde_pad == 0 and all(N % 4 == 0 for M, N, K in shapes if M and N)
        path = "batched fused " + ("tma epilogue" if tma else "staged" if out == "aligned" else "staged scalar")
    else:
        path = "batched " + ("staged" if out == "aligned" else "staged scalar")
    for (M, N, K), q, (C64, scale), (buf, _) in zip(shapes, probs, refs, bufs):
        what = f"batched {M}x{N}x{K} ta={ta} tb={tb} {cls} relu={relu} acc={accumulate} fused={fused} out={out} lde+{lde_pad}"
        if M and N:
            _record(path, cls, q[2], C64, scale, what)
        outside_untouched(buf, q[2], what)
    assert all(torch.equal(a.view(torch.int32), b.view(torch.int32)) for a, b in zip(first, run())), "second call differs"
    return [q[2].clone() for q in probs]


BATCH_SHORT = [(257, 60, 36), (0, 60, 100), (1000, 129, 512), (1, 4, 4), (129, 520, 100), (127, 0, 36)]
BATCH_LONG = BATCH_SHORT[:4] + [(129, 520, 4100), (127, 4, 544)]
BATCH_N4 = [(257, 60, 36), (0, 60, 100), (1000, 128, 512), (1, 4, 4), (129, 520, 100), (127, 0, 36)]   # every N % 4 == 0
BATCH_N4_LONG = BATCH_N4[:4] + [(129, 520, 4100), (127, 4, 544)]


@pytest.mark.parametrize("ta,tb", [(0, 0), (0, 1), (1, 0), (1, 1)])
@pytest.mark.parametrize("relu,accumulate", [(False, False), (True, False), (False, True), (True, True)])
def test_batched(dc, ta, tb, relu, accumulate):
    i = 2 * ta + tb
    for j, shapes in enumerate((BATCH_SHORT, BATCH_LONG)):
        _batched(dc, shapes, bool(ta), bool(tb), CLASSES[(i + j + 2 * relu + accumulate) % len(CLASSES)], relu=relu,
                 accumulate=accumulate, out="ldc" if (i + relu) % 3 == 0 else "aligned", seed=300 + 8 * i + 2 * relu + accumulate)


@pytest.mark.parametrize("ta,tb", [(0, 0), (0, 1), (1, 0), (1, 1)])
@pytest.mark.parametrize("variant", ["tma", "tma long", "ragged", "ragged long", "lde", "scalar"])
def test_batched_fused_epilogue(dc, ta, tb, variant):
    """C = E o (acc - rowv): aligned E and every N % 4 == 0 (TMA epilogue, short and long contractions), a problem with
    N % 4 != 0 in the batch (staged), lde % 4 != 0 (staged, scalar E loads) and C with ldc % 4 != 0 (scalar stores)."""
    i = 2 * ta + tb
    shapes = {"tma": BATCH_N4, "tma long": BATCH_N4_LONG, "ragged long": BATCH_LONG}.get(variant, BATCH_SHORT)
    for cls in ("randn", "relu", "rowcol"):
        _batched(dc, shapes, bool(ta), bool(tb), cls, fused=True, out="ldc" if variant == "scalar" else "aligned",
                 lde_pad=1 if variant == "lde" else 0, seed=400 + 8 * i + CLASSES.index(cls))


@pytest.mark.parametrize("relu,accumulate,fused", [(False, False, False), (True, False, False), (False, True, False),
                                                    (True, True, False), (False, False, True)])
def test_batched_fallback_matches_the_tensor_path(dc, relu, accumulate, fused):
    """The per-problem fallback of ops.gemm_batched (taken when any problem of the batch is unaligned) computes what the
    one-launch tensor path computes, for every combination of epilogues the batched entry point accepts."""
    shapes = [(257, 60, 36), (129, 129, 100), (64, 20, 64)]
    tc = _batched(dc, shapes, False, True, "randn", relu=relu, accumulate=accumulate, fused=fused, seed=500)
    # the same problems, plus an unaligned one (lda % 4 != 0) that sends the whole batch to the fallback
    ops = dc.ops
    g = torch.Generator(device="cuda").manual_seed(501)
    probs, olds = [], []
    for j, (M, N, K) in enumerate(shapes):
        A, B = operands("randn", M, N, K, 500 + 7 * j, device="cuda")
        C = torch.empty(M, N, device="cuda")
        c_old = torch.randn(M, N, generator=g, device="cuda") if accumulate else None
        if accumulate:
            C.copy_(c_old)
        q = (stored(A, False), stored(B, True), C)
        if fused:
            q = q + (torch.rand(((M, (N + 3) // 4 * 4)), generator=g, device="cuda")[:, :N], torch.randn(M, generator=g, device="cuda"))
        probs.append(q)
        olds.append(c_old)
    odd = (torch.randn(8, 21, device="cuda"), torch.randn(8, 21, device="cuda"), torch.empty(8, 8, device="cuda"))
    ops.gemm_batched(probs + [odd], trans_b=True, relu=relu, accumulate=accumulate)
    for q, c_old, c_tc, (M, N, K) in zip(probs, olds, tc, shapes):
        C64, scale = reference([q[:2]], False, True, c_old=c_old, E=q[3] if fused else None, rowv=q[4] if fused else None,
                               relu=relu)
        check_product(q[2], C64, scale, what=f"fallback {M}x{N}x{K} relu={relu} acc={accumulate} fused={fused}")
        assert (q[2] - c_tc).abs().max().item() <= 2e-6 * scale.max().item(), "fallback and tensor path differ"


AUTO = [   # products above the 1e8 work cut, at the shapes the model runs
    (2000, 1200, 512, 0, 1, dict(bias="aligned", relu=True)),     # layer product, >= 148 tiles: TMA epilogue
    (2000, 1200, 544, 0, 1, dict(bias="aligned")),                # the same with K > 512
    (4000, 256, 544, 0, 0, dict(accumulate=True)),                # P Xr-like, split-K
    (256, 256, 4100, 1, 0, {}),                                   # weight gradient dq^T xs: 16 parts
    (20000, 128, 384, 0, 1, dict(bias="misaligned", relu=True)),
]


@pytest.mark.parametrize("M,N,K,ta,tb,epi", AUTO)
def test_auto_dispatch_takes_the_tensor_path(dc, M, N, K, ta, tb, epi):
    cls = "relu" if ta else "randn"
    ours = _single(dc, M, N, (K,), bool(ta), bool(tb), cls, precision=dc.ops.GEMM_AUTO, seed=600 + K, **epi)
    tc = _single(dc, M, N, (K,), bool(ta), bool(tb), cls, seed=600 + K, **epi)
    assert torch.equal(ours, tc), "AUTO did not run the tensor-core kernel"
