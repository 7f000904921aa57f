"""GPU numerics of the tcgen05 linear layer (csrc/gemm.cu) against a plain PyTorch fp32 reference of the
same op (inputs rounded to the 16-bit type first, fp32 math, one rounding of the result).  Tolerance:
the result must be within 1 ulp(16-bit) + 1e-3*|ref| of the correctly rounded fp32 reference — what a
different fp32 accumulation order can cost — and bit-exact on exact-grid inputs."""
import math

import pytest
import torch

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available()
    from atlas_b200._lib import lib

    lib()
    return torch.device("cuda:0")


def _ref(x, w, bias, residual, epi):
    acc = x.float() @ w.float().T
    if epi in (1, 2, 3) and bias is not None:
        acc = acc + bias.float()
    if epi == 2:
        acc = torch.nn.functional.gelu(acc)                       # erf GELU (modeling_bert.py:444)
    if epi == 3:
        acc = acc + residual.float()
    if epi == 4:
        a, b = acc[:, 0::2], acc[:, 1::2]
        acc = torch.nn.functional.gelu(a, approximate="tanh") * b  # gelu_new in fp32 (modeling_t5.py:283)
    return acc


def _close(got, ref, dtype):
    ref16 = ref.to(dtype).float()
    ulp = (torch.finfo(dtype).eps * ref16.abs()).clamp_min(torch.finfo(dtype).tiny * 1024)
    err = (got.float() - ref).abs()
    # 1 ulp of the 16-bit result + relative slack + an ABSOLUTE term for fp32 accumulation-order noise
    # (the fp32 torch reference itself is ~5e-6 away from the fp64 value at K = 3072; measured, tools/diag_gemm.py)
    return bool((err <= 1.0 * ulp + 1e-3 * ref.abs() + 3e-5).all()), float(err.max())


@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16])
@pytest.mark.parametrize("M,N,K", [(128, 128, 64), (257, 768, 768), (1000, 3072, 768), (333, 768, 3072),
                                   (4096, 2304, 768), (19200, 768, 768), (64, 32128, 768),
                                   (9999, 1032, 520)])   # 256 x 256 CTA-pair tiles with ragged M / N / K tails
@pytest.mark.parametrize("epi", [0, 1, 2, 3])
def test_linear_matches_fp32_reference(dev, dtype, M, N, K, epi):
    from atlas_b200 import ops

    g = torch.Generator(device="cpu").manual_seed(M * 7 + N * 3 + K + epi)
    x = (torch.randn(M, K, generator=g) * 0.5).to(dtype).to(dev)
    w = (torch.randn(N, K, generator=g) / math.sqrt(K)).to(dtype).to(dev)
    bias = (torch.randn(N, generator=g) * 0.1).to(dtype).to(dev)
    res = (torch.randn(M, N, generator=g)).to(dtype).to(dev)
    y = ops.linear(x, w, bias if epi else None, res if epi == 3 else None, epilogue=epi)
    ok, err = _close(y, _ref(x, w, bias, res, epi), dtype)
    assert ok, f"max abs err {err}"


@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16])
@pytest.mark.parametrize("M", [777, 5000])      # 1-CTA tiles / 2-CTA pair tiles
def test_gated_gelu_epilogue(dev, dtype, M):
    from atlas_b200 import ops

    g = torch.Generator(device="cpu").manual_seed(5)
    K, F = 768, 2048
    x = (torch.randn(M, K, generator=g) * 0.5).to(dtype).to(dev)
    w0 = (torch.randn(F, K, generator=g) / math.sqrt(K)).to(dtype)
    w1 = (torch.randn(F, K, generator=g) / math.sqrt(K)).to(dtype)
    w = torch.stack([w0, w1], dim=1).reshape(2 * F, K).contiguous().to(dev)   # rows interleaved wi_0 / wi_1
    y = ops.linear(x, w, epilogue=ops.EPI_GATED)
    assert y.shape == (M, F)
    ok, err = _close(y, _ref(x, w, None, None, 4), dtype)
    assert ok, f"max abs err {err}"


def test_exact_grid_bit_exact(dev):
    """Inputs on a coarse grid: every partial sum is exact in fp32, so the result must equal the fp32
    reference bit for bit after the single rounding."""
    from atlas_b200 import ops

    g = torch.Generator(device="cpu").manual_seed(9)
    x = (torch.randint(-8, 9, (515, 768), generator=g).float() / 8).half().to(dev)
    w = (torch.randint(-8, 9, (1536, 768), generator=g).float() / 8).half().to(dev)
    y = ops.linear(x, w)
    assert torch.equal(y, (x.float() @ w.float().T).half())


def test_strided_input_and_output_view(dev):
    from atlas_b200 import ops

    g = torch.Generator(device="cpu").manual_seed(11)
    big = (torch.randn(300, 2304, generator=g) * 0.3).half().to(dev)
    x = big[:, 768:1536]                                   # row stride 2304, K = 768
    w = (torch.randn(768, 768, generator=g) / 27.7).half().to(dev)
    out = torch.zeros(300, 1536, dtype=torch.float16, device=dev)
    ops.linear(x, w, out=out[:, 768:])
    ok, err = _close(out[:, 768:], x.float() @ w.float().T, torch.float16)
    assert ok and float(out[:, :768].abs().max()) == 0.0


@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16])
@pytest.mark.parametrize("M", [300, 6000])      # 1-CTA tiles / 2-CTA pair tiles
def test_fused_rmsnorm_around_the_gemm(dev, dtype, M):
    """atlas_b200_linear_ex: (a) `out_ss` = sum of squares of the stored residual output rows, (b) `row_ss` scales the
    accumulator rows by rsqrt(ss / K + eps) - together T5's RMSNorm (src/modeling_t5.py:244-253) with the norm weight
    folded into the consumer's matrix.  Reference: fp32 torch of the same folded computation, and the un-fused
    layernorm + linear path of this library (same result up to the 16-bit rounding of the normalised activations)."""
    from atlas_b200 import ops

    g = torch.Generator(device="cpu").manual_seed(11 + M)
    d, F = 768, 1024
    ctx = (torch.randn(M, d, generator=g) * 0.5).to(dtype).to(dev)
    wo = (torch.randn(d, d, generator=g) / math.sqrt(d)).to(dtype).to(dev)
    res = (torch.randn(M, d, generator=g) * 3.0).to(dtype).to(dev)
    ln = (1.0 + 0.1 * torch.randn(d, generator=g)).to(dtype).to(dev)
    wi = (torch.randn(F, d, generator=g) / math.sqrt(d)).to(dtype).to(dev)
    eps = 1e-6
    ss = torch.zeros(M, dtype=torch.float32, device=dev)
    h = ops.linear(ctx, wo, None, residual=res, epilogue=ops.EPI_RESIDUAL, out_ss=ss)
    h_plain = ops.linear(ctx, wo, None, residual=res, epilogue=ops.EPI_RESIDUAL)
    assert torch.equal(h, h_plain)
    ss_ref = h.float().pow(2).sum(-1)
    assert torch.allclose(ss, ss_ref, rtol=2e-5, atol=1e-4), float((ss - ss_ref).abs().max())
    wi_n = (wi.float() * ln.float()[None, :]).to(dtype)
    y = ops.linear(h, wi_n, row_ss=ss, rs_eps=eps)
    ref = (h.float() @ wi_n.float().T) * torch.rsqrt(ss_ref / d + eps)[:, None]
    ok, err = _close(y, ref, dtype)
    assert ok, f"max abs err {err}"
    # against the un-fused path (normalised activations rounded to 16 bits in between): same up to that rounding
    y2 = ops.linear(ops.layernorm(h, ln, None, eps, kind=1), wi)
    tol = 4 * torch.finfo(dtype).eps
    assert float((y.float() - y2.float()).abs().max()) <= tol * float(y2.float().abs().max()) + 1e-3


@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16])
@pytest.mark.parametrize("M,N,K,epi", [
    (30720, 2304, 768, 0),      # FiD-base fused q|k|v projection of 2 queries x 40 passages
    (30720, 768, 2048, 3),      # wo + residual
    (20580, 768, 768, 3),       # M = 40 x 512 + 100: the second pair of the last cluster is entirely out of range
    (20780, 1032, 520, 1),      # M = 40 x 512 + 300: ... partly out of range; ragged N and K
    (16384, 4096, 768, 4),      # gated-GELU epilogue
])
def test_quad_cluster_multicast_tiles(dev, dtype, M, N, K, epi, tmp_path):
    """Shapes large enough for the 4-CTA-cluster kernel (two CTA pairs sharing the W tile through TMA multicast): against the
    fp32 reference, and bit-identical to the 2-CTA pair kernel (same MMA order per output element: the accumulation over K
    is the same sequence of UMMA K = 16 steps in both)."""
    import os
    import subprocess
    import sys

    from atlas_b200 import ops

    g = torch.Generator(device="cpu").manual_seed(M + N + K + epi)
    x = (torch.randn(M, K, generator=g) * 0.5).to(dtype).to(dev)
    w = (torch.randn(N, K, generator=g) / math.sqrt(K)).to(dtype).to(dev)
    bias = (torch.randn(N, generator=g) * 0.1).to(dtype).to(dev)
    res = (torch.randn(M, N, generator=g)).to(dtype).to(dev)
    y = ops.linear(x, w, bias if epi in (1, 2, 3) else None, res if epi == 3 else None, epilogue=epi)
    ok, err = _close(y, _ref(x, w, bias, res, epi), dtype)
    assert ok, f"max abs err {err}"
    # the quad-cluster kernel in a child process (the switch is read once per process; the default is the pair kernel)
    code = (
        "import sys, math, torch; sys.path.insert(0, %r)\n"
        "from atlas_b200 import ops\n"
        "M, N, K, epi, dt = %d, %d, %d, %d, torch.%s\n"
        "g = torch.Generator(device='cpu').manual_seed(M + N + K + epi)\n"
        "dev = torch.device('cuda:0')\n"
        "x = (torch.randn(M, K, generator=g) * 0.5).to(dt).to(dev)\n"
        "w = (torch.randn(N, K, generator=g) / math.sqrt(K)).to(dt).to(dev)\n"
        "bias = (torch.randn(N, generator=g) * 0.1).to(dt).to(dev)\n"
        "res = (torch.randn(M, N, generator=g)).to(dt).to(dev)\n"
        "y = ops.linear(x, w, bias if epi in (1, 2, 3) else None, res if epi == 3 else None, epilogue=epi)\n"
        "torch.save(y.cpu(), sys.argv[1])\n"
    ) % (os.path.dirname(os.path.dirname(os.path.abspath(__file__))), M, N, K, epi, str(dtype).split(".")[1])
    path = str(tmp_path / "quad.pt")
    env = dict(os.environ, ATLAS_B200_GEMM_QUAD="1")     # the child runs the opt-in quad-cluster kernel
    subprocess.run([sys.executable, "-c", code, path], check=True, env=env, timeout=300)
    y_quad = torch.load(path)
    assert torch.equal(y.cpu(), y_quad), "the quad-cluster kernel and the pair kernel disagree"
