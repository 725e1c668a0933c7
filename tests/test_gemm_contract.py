"""The GEMM accuracy contract (tests/gemm_contract.py) can fail: a CPU emulation of K2's split and tensor-core accumulator
passes both bounds with room to spare, and each plausible degraded split fails at least one input class by 2x or more.

The emulation follows csrc/gemm_tc2.cu:
  * hi = the raw fp32 operand truncated to tf32 (the tensor core ignores the low 13 bits); lo = x - hi (exact in fp32),
    pre-biased by 0x1000 on its bit pattern so that the tensor core's truncation rounds it to nearest;
  * every 8-deep MMA adds its exact products to an fp32 accumulator rounded towards zero; main (hi hi) and cross
    (hi lo, then lo hi: two MMAs) accumulate separately, in chains of 4 * drain_kb MMAs;
  * a drained chain is added in fp32 round-to-nearest: acc = fmaf(main, 1 + comp * n, acc); acc += cross.
Degraded variants: single-pass TF32, two terms (lo hi dropped), 3xBF16, 3xFP16 with one power-of-two scale per matrix, and
K2 with chains of 32 k-blocks and no compensation (DCB200_DRAIN_KB=32 DCB200_T2_COMP=0)."""
import pytest
import torch

from gemm_contract import CLASSES, TAU_ELEM, TAU_GLOBAL, measure, operands, reference

M, N, K = 96, 96, 2048
DRAIN_KB, COMP = 4, 2.6e-8          # T2_DRAIN_KB, t2_numerics() defaults


def _tf32_trunc(x):
    return (x.view(torch.int32) & -8192).view(torch.float32)


def _tf32_biased(x):                # the kernel's lo: + 0x1000 on the bit pattern, then the tensor core's truncation
    return ((x.view(torch.int32) + 0x1000) & -8192).view(torch.float32)


def _rz32(x):                       # float64 -> fp32 rounded towards zero
    f = x.float()
    return torch.where(f.double().abs() > x.abs(), torch.nextafter(f, torch.zeros_like(f)), f)


def _split_k2(A, B):
    ah, bh = _tf32_trunc(A), _tf32_trunc(B)
    return ah, _tf32_biased(A - ah), bh, _tf32_biased(B - bh), 1.0


def _split_bf16(A, B):
    bf = lambda x: x.bfloat16().float()
    ah, bh = bf(A), bf(B)
    return ah, bf(A - ah), bh, bf(B - bh), 1.0


def _split_fp16_scaled(A, B):
    sa = 2.0 ** (14 - torch.ceil(torch.log2(A.abs().max())).item())
    sb = 2.0 ** (14 - torch.ceil(torch.log2(B.abs().max())).item())
    hf = lambda x: x.half().float()
    As, Bs = A * sa, B * sb
    ah, bh = hf(As), hf(Bs)
    return ah, hf(As - ah), bh, hf(Bs - bh), 1.0 / (sa * sb)


def _split_tf32_once(A, B):
    return _tf32_biased(A), torch.zeros_like(A), _tf32_biased(B), torch.zeros_like(B), 1.0


def tc_product(A, B, split=_split_k2, drain_kb=DRAIN_KB, comp=COMP, terms=3):
    """Emulated tensor-core product of fp32 A [M, K] and B [K, N] (see the module docstring)."""
    ah, al, bh, bl, unscale = split(A, B)
    ah, al, bh, bl = ah.double(), al.double(), bh.double(), bl.double()
    acc = torch.zeros(A.shape[0], B.shape[1], dtype=torch.float32)
    K_ = A.shape[1]
    chain = 8 * 4 * drain_kb
    for c0 in range(0, K_, chain):
        main = torch.zeros_like(acc)
        cross = torch.zeros_like(acc)
        c1 = min(K_, c0 + chain)
        for k0 in range(c0, c1, 8):
            s = slice(k0, k0 + 8)
            main = _rz32(main.double() + ah[:, s] @ bh[s])
            cross = _rz32(cross.double() + ah[:, s] @ bl[s])
            if terms == 3:
                cross = _rz32(cross.double() + al[:, s] @ bh[s])
        # the epilogue's factor counts 4 MMAs per (32-deep) k-block of the chain, in fp32 like the kernel's
        n = 4 * ((c1 - c0 + 31) // 32)
        f = torch.tensor(1.0, dtype=torch.float32) + torch.tensor(comp, dtype=torch.float32) * n
        acc = (acc.double() + main.double() * f.double()).float()     # fmaf: one rounding
        acc = acc + cross
    return (acc.double() * unscale).float()


VARIANTS = {
    "tf32 single pass": dict(split=_split_tf32_once),
    "2 terms": dict(terms=2),
    "3xBF16": dict(split=_split_bf16),
    "3xFP16 per-matrix scale": dict(split=_split_fp16_scaled),
    "drain 32 k-blocks, no comp": dict(drain_kb=32, comp=0.0),
}


def _run(cls, **kw):
    A, B = operands(cls, M, N, K, seed=CLASSES.index(cls))
    C64, scale = reference([(A, B)], ta=False, tb=False)
    elem, _, glob = measure(tc_product(A, B, **kw), C64, scale)
    return elem, glob


@pytest.fixture(scope="module")
def k2():
    return {cls: _run(cls) for cls in CLASSES}


def test_emulated_k2_meets_the_contract_with_2x_margin(k2):
    for cls, (elem, glob) in k2.items():
        assert elem <= TAU_ELEM / 2 and glob <= TAU_GLOBAL / 2, f"{cls}: elementwise {elem:.2e}, global {glob:.2e}"


def test_exact_data_is_exact_without_compensation():
    """ints: C64 is exact, so the only error left is the compensation factor (1 + comp * n)."""
    A, B = operands("ints", M, N, K, seed=0)
    C64, scale = reference([(A, B)], ta=False, tb=False)
    assert torch.equal(tc_product(A, B, comp=0.0).double(), C64)


@pytest.mark.parametrize("variant", list(VARIANTS))
def test_degraded_split_fails_the_contract(variant):
    worst = max(max(e / TAU_ELEM, g / TAU_GLOBAL) for e, g in (_run(cls, **VARIANTS[variant]) for cls in CLASSES))
    assert worst >= 2.0, f"{variant}: worst class at {worst:.2f}x the bounds (needs >= 2x to be rejected reliably)"


@pytest.mark.parametrize("relu,accumulate", [(True, False), (False, True), (True, True)])
def test_fused_epilogue_excludes_relu_and_accumulate(relu, accumulate):
    """dc_gemm_batched and ops.gemm_batched reject a fused epilogue operand E together with relu or accumulate, before any
    device work (the tensor-core path and the per-problem fallback would otherwise compose them in different orders)."""
    from deformcontact_b200 import _abi, ops
    A, B, Cm, E, rowv = torch.zeros(8, 4), torch.zeros(8, 4), torch.zeros(8, 8), torch.zeros(8, 8), torch.zeros(8)
    with pytest.raises(_abi.DcError, match="excludes relu and accumulate"):
        ops.gemm_batched([(A, B, Cm), (A, B, Cm, E, rowv)], relu=relu, accumulate=accumulate)
    arr = (_abi.GemmProblem * 2)()
    for i in range(2):   # host addresses: the entry point must refuse before it reads any of them
        arr[i] = _abi.GemmProblem(A.data_ptr(), 4, B.data_ptr(), 4, Cm.data_ptr(), 8, 8, 8, 4,
                                  E.data_ptr() if i else None, 8 if i else 0, rowv.data_ptr() if i else None)
    with pytest.raises(_abi.DcError, match=f"status {_abi.DC_EINVAL}:.*excludes relu and accumulate"):
        _abi.call("dc_gemm_batched", arr, 2, 0, 1, int(relu), int(accumulate), None, 0, None, 0, None)
