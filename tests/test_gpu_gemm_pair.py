"""-m gpu: the CTA-pair GEMM (csrc/gemm_tcgen05.cu, gemm_bf16_tcgen05_pair_kernel: a cluster of two CTAs per 256 x 256 tile,
tcgen05.mma.cta_group::2) against the single-CTA kernel it replaces on large problems and against torch.
Same products, same k order, fp32 accumulation in TMEM: the two kernels must agree bit for bit.

The single-CTA reference is the pinned ``tile_n=256`` (split_k 0 = no K split).  It is the kernel gemm_bf16's own ladder picks
for every shape below when the pair kernel is left out: on the 148 SMs of a B200 each has N >= 256 and
ceil(M / 128) * ceil(N / 256) >= 148 tiles (150, 3840, 745, 1413 and 891 for the plain shapes, 3000 for the epilogue shape),
so it runs 256-wide tiles without split-K."""
import pytest
import torch

pytestmark = pytest.mark.gpu


def _ops():
    from importlib import import_module
    import fo1_b200  # noqa: F401
    return import_module("vlm-fo1_b200.ops")


def _both(fn):
    """fn(tile_n): the library's choice (the pair kernel), then the single-CTA kernel pinned to 256-wide tiles."""
    a = fn(0)
    torch.cuda.synchronize()
    b = fn(256)
    torch.cuda.synchronize()
    return a, b


@pytest.mark.parametrize("M,N,K", [(19200, 256, 64), (32768, 3840, 1280), (19000, 1280, 3456), (20000, 2304, 256), (37888 + 77, 520, 1280)])
def test_pair_equals_single_cta_plain(M, N, K):
    ops = _ops()
    g = torch.Generator(device="cuda").manual_seed(M + N)
    a = (torch.randn(M, K, device="cuda", generator=g) * 0.5).bfloat16()
    w = (torch.randn(N, K, device="cuda", generator=g) * 0.05).bfloat16()
    x, y = _both(lambda t: ops.gemm(a, w, tile_n=t))
    assert torch.equal(x, y)
    rows = torch.randint(0, M, (64,), device="cuda")
    ref = (a[rows].float() @ w.float().t())
    assert float((x[rows].float() - ref).abs().max()) <= 2.0 ** -7 * float(ref.abs().max()) + 1e-3


def test_pair_equals_single_cta_epilogues():
    ops = _ops()
    g = torch.Generator(device="cuda").manual_seed(7)
    M, N, K = 38400, 2560, 1280
    a = (torch.randn(M, K, device="cuda", generator=g) * 0.5).bfloat16()
    w = (torch.randn(N, K, device="cuda", generator=g) * 0.05).bfloat16()
    bias = (torch.randn(N, device="cuda", generator=g) * 0.1).bfloat16()
    res = torch.randn(M, N, device="cuda", generator=g).bfloat16()
    x, y = _both(lambda t: ops.gemm(a, w, bias=bias, act="gelu", residual=res, tile_n=t))
    assert torch.equal(x, y)
    x, y = _both(lambda t: ops.gemm(a, w, bias=bias, act="silu", gated=True, tile_n=t))
    assert torch.equal(x, y)
    x, y = _both(lambda t: ops.gemm(a, w, out_dtype=torch.float32, tile_n=t))
    assert torch.equal(x, y)
