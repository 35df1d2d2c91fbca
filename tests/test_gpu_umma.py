"""Pins the tcgen05/TMA operand layouts (shared-memory descriptors, swizzle modes, TMA boxes) used by the bf16
kernels against a plain matmul, through the stgcn_umma_selftest entry point."""
import pytest
import torch

pytestmark = pytest.mark.gpu


def _run(mode, A, B, M, N, K, lbo_a=0, sbo_a=0, lbo_b=0, sbo_b=0):
    from stgcn_b200 import _lib as L
    C = torch.full((M, N), float("nan"), device=A.device, dtype=torch.float32)
    L.check(L.lib().stgcn_umma_selftest(mode, A.data_ptr(), B.data_ptr(), C.data_ptr(), M, N, K, lbo_a, sbo_a, lbo_b,
                                        sbo_b, torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    return C


def _err(C, ref):
    if not torch.isfinite(C).all():
        return float("inf")
    return float((C - ref).abs().max() / ref.abs().max())


@pytest.mark.parametrize("M,N,K", [(128, 128, 64), (256, 128, 192), (128, 16, 64), (128, 64, 128), (128, 256, 64)])
def test_k_major_sw128(M, N, K, cuda_device):
    g = torch.Generator(device="cpu").manual_seed(M + N + K)
    A = torch.randn(M, K, generator=g).to(cuda_device).bfloat16()
    B = torch.randn(N, K, generator=g).to(cuda_device).bfloat16()
    C = _run(0, A, B, M, N, K)
    assert _err(C, A.float() @ B.float().T) < 1e-3


@pytest.mark.parametrize("M,N,K", [(128, 128, 16), (256, 128, 48), (128, 16, 48)])
def test_k_major_sw32(M, N, K, cuda_device):
    g = torch.Generator(device="cpu").manual_seed(M + N + K)
    A = torch.randn(M, K, generator=g).to(cuda_device).bfloat16()
    B = torch.randn(N, K, generator=g).to(cuda_device).bfloat16()
    C = _run(1, A, B, M, N, K)
    assert _err(C, A.float() @ B.float().T) < 1e-3


def test_mn_major_layout_probe(cuda_device):
    """Sweeps the LBO/SBO hypotheses for the MN-major modes, prints the table and asserts the assignment the
    production kernels use."""
    g = torch.Generator(device="cpu").manual_seed(7)
    lines = []
    # mode 2: A [K,M], B [K,N], 128B swizzle, 64-element chunks
    M, N, K = 128, 128, 128
    A = torch.randn(K, M, generator=g).to(cuda_device).bfloat16()
    B = torch.randn(K, N, generator=g).to(cuda_device).bfloat16()
    ref = A.float().T @ B.float()
    res2 = {}
    for lbo, sbo in [(8192, 1024), (1024, 8192)]:
        res2[(lbo, sbo)] = _err(_run(2, A, B, M, N, K, lbo, sbo, lbo, sbo), ref)
        lines.append(f"mode2 lbo={lbo} sbo={sbo} err={res2[(lbo, sbo)]:.3e}")
    # mode 3: A [M,K] K-major; B [G][K][16] MN-major 32B swizzle
    M, G, K = 128, 8, 128
    N = 16 * G
    A3 = torch.randn(M, K, generator=g).to(cuda_device).bfloat16()
    B3 = torch.randn(G, K, 16, generator=g).to(cuda_device).bfloat16()
    ref3 = torch.einsum("mk,gkc->mgc", A3.float(), B3.float()).reshape(M, N)
    res3 = {}
    for lbo, sbo in [(2048, 256), (256, 2048)]:
        res3[(lbo, sbo)] = _err(_run(3, A3, B3, M, N, K, 0, 0, lbo, sbo), ref3)
        lines.append(f"mode3 lbo_b={lbo} sbo_b={sbo} err={res3[(lbo, sbo)]:.3e}")
    print("\n".join(lines))
    assert res2[(8192, 1024)] < 1e-3, lines
    assert res3[(2048, 256)] < 1e-3, lines
