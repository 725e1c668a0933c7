"""Accuracy contract of the tensor-core GEMM (K2, csrc/gemm_tc2.cu; DESIGN.md section 3): shared helpers, not a conftest.

A product C of fp32 operands must satisfy, against the float64 product C64 of the same fp32 inputs, BOTH

    elementwise   |C - C64|_ij <= TAU_ELEM * scale_ij      scale = |opA(A)| |opB(B)|  (+ |bias| + |C_old|, times |E|)
    global        max |C - C64| / max |C64| <= TAU_GLOBAL

The elementwise bound is the one that sees small rows and columns: the global metric is normalised by the largest element
of the whole output, so rows orders of magnitude smaller than the largest can be completely wrong and still pass it.

The input classes are the operand shapes the model actually multiplies: random signs (``randn``), sign-coherent operands
(``relu``: P Xr, P^T dO, dW = dq^T xs), rows and columns of very different scale (``rowcol``), K-blocks of different scale
(``kblock``: concatenated segments such as the decoder input), exact small integers where C64 is exact (``ints``), and zero
rows / columns with a one-hot B (``sparse``)."""
import torch

# >= 2x the worst value measured on the B200 over every path and class: 7.8e-7 and 9.9e-7 (DESIGN.md section 3)
TAU_ELEM = 1.6e-6
TAU_GLOBAL = 2e-6

CLASSES = ("randn", "relu", "rowcol", "kblock", "ints", "sparse")


def operands(cls, M, N, K, seed, device="cpu"):
    """Logical fp32 operands opA [M, K] and opB [K, N] of input class ``cls``, seeded."""
    g = torch.Generator(device=device).manual_seed(seed)
    rn = lambda *s: torch.randn(*s, generator=g, device=device)
    ex = lambda lo, hi, *s: torch.exp2(lo + (hi - lo) * torch.rand(*s, generator=g, device=device))
    if cls == "randn":
        return rn(M, K), rn(K, N)
    if cls == "relu":
        return rn(M, K).relu(), rn(K, N).relu()
    if cls == "rowcol":
        return rn(M, K) * ex(-20, 20, M, 1), rn(K, N) * ex(-20, 20, 1, N)
    if cls == "kblock":   # blocks of 24 contraction indices (not aligned with the kernel's 32-wide k-blocks)
        s = ex(-12, 12, (K + 23) // 24).repeat_interleave(24)[:K]
        return rn(M, K) * s[None, :], rn(K, N)
    if cls == "ints":
        return (torch.randint(-2, 3, (M, K), generator=g, device=device).float(),
                torch.randint(-2, 3, (K, N), generator=g, device=device).float())
    if cls == "sparse":
        A = rn(M, K) * (torch.rand(M, 1, generator=g, device=device) > 0.2)          # ~20 % zero rows
        B = torch.zeros(K, N, device=device)
        B[torch.randint(0, K, (N,), generator=g, device=device), torch.arange(N, device=device)] = 1.0
        return A, B * (torch.rand(1, N, generator=g, device=device) > 0.2)             # one-hot columns, ~20 % zero
    raise ValueError(cls)


def stored(X, trans):
    """X ([rows, cols] logical) stored as the GEMM reads it: ``X`` itself or, with ``trans``, a [cols, rows] tensor whose
    transpose is X.  Rows are padded to a multiple of 4 floats (16-byte pitch) and the result is a view."""
    Y = X.t() if trans else X
    r, c = Y.shape
    buf = torch.empty((r, (c + 3) // 4 * 4), dtype=X.dtype, device=X.device)
    buf[:, :c] = Y
    return buf[:, :c]


def reference(segs, ta=False, tb=True, bias=None, c_old=None, E=None, rowv=None, relu=False):
    """float64 reference of ``ops.gemm`` / ``ops.gemm_batched`` on the device of the operands:
    C64 = act(E o (sum_s opA(A_s) opB(B_s) + bias - rowv[:, None]) + C_old) and the scale of the elementwise bound."""
    C64, scale = 0.0, 0.0
    for A, B in segs:
        a = A.double().t() if ta else A.double()
        b = B.double().t() if tb else B.double()
        C64 = C64 + a @ b
        scale = scale + a.abs() @ b.abs()
    if bias is not None:
        C64, scale = C64 + bias.double(), scale + bias.double().abs()
    if E is not None:
        C64 = E.double() * (C64 - rowv.double()[:, None])
        scale = E.double().abs() * (scale + rowv.double().abs()[:, None])
    if c_old is not None:
        C64, scale = C64 + c_old.double(), scale + c_old.double().abs()
    if relu:
        C64 = C64.relu()
    return C64, scale


def measure(C, C64, scale):
    """(worst elementwise ratio, its (row, col), global metric).  Where the scale is 0 the result must be exact."""
    err = (C.double() - C64).abs()
    ratio = torch.where(scale > 0, err / scale.clamp_min(1e-300), torch.where(err > 0, float("inf"), 0.0))
    flat = int(ratio.argmax()) if C.numel() else 0
    ij = (flat // C.shape[1], flat % C.shape[1]) if C.numel() else (0, 0)
    top = C64.abs().max().item() if C.numel() else 0.0
    emax = err.max().item() if C.numel() else 0.0
    glob = emax / top if top > 0 else (0.0 if emax == 0 else float("inf"))
    return (ratio.max().item() if C.numel() else 0.0), ij, glob


SENTINEL = 0x7FBADBAD          # a NaN payload no kernel writes


def sentinel_out(M, N, ld, offset, device="cuda"):
    """(buffer, C): C [M, N] with row pitch ``ld`` at element ``offset`` of an fp32 buffer filled with the SENTINEL bit pattern,
    which extends at least one row past C at both ends; ``offset % 4`` is C's distance in floats from a 16-byte boundary."""
    buf = torch.full((offset + (M + 1) * ld + N,), SENTINEL, dtype=torch.int32, device=device).view(torch.float32)
    return buf, buf.as_strided((M, N), (ld, 1), offset)


def outside_untouched(buf, C, what):
    """Every element of ``buf`` that is not part of the view ``C`` still holds the sentinel."""
    mask = torch.ones(buf.shape, dtype=torch.bool, device=buf.device)
    mask.as_strided(C.shape, C.stride(), C.storage_offset()).fill_(False)
    assert bool((buf.view(torch.int32)[mask] == SENTINEL).all()), f"{what}: wrote outside C"


def epilogue_path(M, N, kb_total, C, bias, accumulate):
    """The epilogue K2 takes for a single product (gemm_tc2.cu: t2_k_parts, t2_tepi_ok, vec_ok), for the record."""
    sms = torch.cuda.get_device_properties(C.device).multi_processor_count
    tiles = -(-M // 128) * -(-N // 128)
    parts = 1 if tiles >= sms else max(1, min(sms // tiles, kb_total // 8, 64))
    aligned = C.stride(0) % 4 == 0 and C.data_ptr() % 16 == 0
    if parts > 1:
        return "split-k"
    if not accumulate and aligned and N % 4 == 0:
        return "tma epilogue"
    vec = aligned and (bias is None or bias.data_ptr() % 16 == 0)
    return "staged" if vec else "staged scalar"


def check_product(C, C64, scale, tau_elem=TAU_ELEM, tau_global=TAU_GLOBAL, what=""):
    """Assert both bounds; returns (elementwise, global) for the record."""
    elem, (i, j), glob = measure(C, C64, scale)
    assert elem <= tau_elem, (f"{what}: elementwise |C - C64| / (|A||B|) = {elem:.3e} > {tau_elem:.1e} at [{i}, {j}]: "
                              f"C = {C[i, j].item()!r}, C64 = {C64[i, j].item()!r}, scale = {scale[i, j].item():.6e}")
    assert glob <= tau_global, f"{what}: max|C - C64| / max|C64| = {glob:.3e} > {tau_global:.1e}"
    return elem, glob
