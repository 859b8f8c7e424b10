"""GPU parity: hand-written tcgen05 GEMM (C ABI sb_gemm_bf16_tn) vs a plain PyTorch fp32 reference
computed on the SAME bf16-rounded operands (so the only difference is accumulation order)."""
import pytest
import torch

pytestmark = pytest.mark.gpu


def _gemm(A, B, bias=None, accumulate_into=None, split_k=1, remap=None):
    from speech_b200 import _lib
    lib = _lib.load()
    M, K = A.shape
    N = B.shape[0]
    flags = 0
    if remap is None:
        C = accumulate_into if accumulate_into is not None else torch.empty(M, N, device="cuda")
        rB = rT = vB = 0
    else:
        rB, rT, vB = remap
        C = torch.zeros(vB * rT, N, device="cuda")
        flags |= 2
    if accumulate_into is not None:
        flags |= 1
    _lib.check(lib.sb_gemm_bf16_tn(A.data_ptr(), A.stride(0), B.data_ptr(), B.stride(0),
                                   C.data_ptr(), C.stride(0), _lib.ptr(bias), M, N, K, flags,
                                   split_k, rB, rT, vB, _lib.stream_ptr()), "gemm")
    torch.cuda.synchronize()
    return C


@pytest.mark.parametrize("M,N,K", [
    (128, 256, 64),       # exactly one tile, one k-block
    (128, 32, 128),
    (256, 512, 256),
    (300, 200, 72),       # ragged everything (K % 64 != 0, partial tiles)
    (15808, 96, 480),     # layer-0 input projection shape class
    (1000, 6144, 2048),   # many tiles per CTA -> ring + TMEM double buffering wrap around
    (4096, 29, 2048),     # output projection N=29 (ldc not a multiple of 4 -> scalar stores)
    (16000, 3072, 1024),  # long-K, many tiles -> CTA-pair kernel (cta_group::2, 256x256 tiles)
    (15808, 6144, 1088),  # same, ragged K (17 k-blocks) and ragged M (15808 = 61.75 x 256)
    (9999, 2100, 1024),   # CTA-pair kernel with ragged M and N (second CTA partly out of range)
    (192, 48, 160),       # tests/shared.py tiny config
])
def test_gemm_matches_fp32_reference(cuda_lib, M, N, K):
    torch.manual_seed(M + N + K)
    A = torch.randn(M, K, device="cuda").bfloat16()
    B = torch.randn(N, K, device="cuda").bfloat16()
    bias = torch.randn(N, device="cuda")
    C = _gemm(A, B, bias)
    ref = A.float() @ B.float().t() + bias
    err = (C - ref).abs().max().item()
    assert err < 2e-3 * (K ** 0.5), err


def test_gemm_split_k_accumulate(cuda_lib):
    torch.manual_seed(0)
    M, N, K = 384, 640, 15808
    A = torch.randn(M, K, device="cuda").bfloat16()
    B = torch.randn(N, K, device="cuda").bfloat16()
    C0 = torch.randn(M, N, device="cuda")
    C = _gemm(A, B, None, accumulate_into=C0.clone(), split_k=4)
    ref = C0 + A.float() @ B.float().t()
    assert (C - ref).abs().max().item() < 0.5
    assert ((C - ref).abs().max() / ref.abs().max()).item() < 1e-4


@pytest.mark.parametrize("M,N,K,split", [
    (1024, 1024, 4096, 1),    # CTA-pair kernel, wave-filling K split chosen by the library
    (6144, 2048, 16000, 2),   # north-star dW_ih shape (the caller's split is only a hint)
    (1000, 700, 5000, 3),     # ragged M, N, K
])
def test_gemm_pair_accumulate_with_library_chosen_split(cuda_lib, M, N, K, split):
    torch.manual_seed(M + K)
    A = torch.randn(M, K, device="cuda").bfloat16()
    B = torch.randn(N, K, device="cuda").bfloat16()
    bias = torch.randn(N, device="cuda")
    C0 = torch.randn(M, N, device="cuda")
    C = _gemm(A, B, bias, accumulate_into=C0.clone(), split_k=split)
    ref = C0 + A.float() @ B.float().t() + bias
    assert ((C - ref).abs().max() / ref.abs().max()).item() < 1e-4


def test_gemm_pair_kernel_is_bit_identical_to_single_cta(cuda_lib):
    """Same k order, same accumulator precision: the cta_group::2 kernel must reproduce the
    single-CTA kernel bit for bit on a plain (non-accumulating) GEMM.  N = 2048 goes to the pair
    kernel; the same product computed as 16 column blocks of N = 128 goes to the single-CTA kernel
    (TMA-store epilogue) block by block."""
    torch.manual_seed(7)
    A = torch.randn(5000, 1536, device="cuda").bfloat16()
    B = torch.randn(2048, 1536, device="cuda").bfloat16()
    bias = torch.randn(2048, device="cuda")
    C1 = torch.cat([_gemm(A, B[j:j + 128], bias[j:j + 128]) for j in range(0, 2048, 128)], 1)
    C2 = _gemm(A, B, bias)
    assert torch.equal(C1, C2)


def test_gemm_row_remap_time_major_to_batch_first(cuda_lib):
    torch.manual_seed(1)
    T, Bp, Bv, K, N = 37, 8, 5, 128, 29
    A = torch.randn(T * Bp, K, device="cuda").bfloat16()
    B = torch.randn(N, K, device="cuda").bfloat16()
    C = _gemm(A, B, None, remap=(Bp, T, Bv))
    ref = (A.float() @ B.float().t()).view(T, Bp, N)[:, :Bv].transpose(0, 1).reshape(Bv * T, N)
    assert (C - ref).abs().max().item() < 2e-2


@pytest.mark.parametrize("M,N,K", [
    (128, 64, 64),        # one tile, one k-block
    (300, 200, 1000),     # ragged everything
    (32, 2048, 15808),    # fc weight gradient shape class (M_out = padded vocabulary)
    (1280, 32, 30000),    # conv weight gradient (transposed form): long K, narrow N
    (3072, 480, 15808),   # layer-0 dW_ih: CTA-pair kernel, split chosen by the library
    (2048, 1024, 15744),  # dW_hh (r,z rows)
])
@pytest.mark.parametrize("a_mn,b_mn", [(True, False), (False, True), (True, True)])
def test_gemm_mn_major_operands_bit_identical_to_k_major(cuda_lib, M, N, K, a_mn, b_mn):
    """MN-major UMMA operands (the contraction runs over the ROWS of the matrix in memory) must
    give exactly the K-major result: same k order, same accumulator, only the shared-memory layout
    and the descriptors differ.  The transposed operands are strided views of wider matrices, as
    the weight-gradient call sites pass them."""
    from speech_b200 import ops
    torch.manual_seed(M + N + K)
    A = torch.randn(M, K, device="cuda").bfloat16()
    B = torch.randn(N, K, device="cuda").bfloat16()
    Mp, Np = (M + 7) // 8 * 8 + 8, (N + 7) // 8 * 8 + 16
    At = torch.zeros(K, Mp, device="cuda", dtype=torch.bfloat16)
    At[:, 8:8 + M] = A.t()
    Bt = torch.zeros(K, Np, device="cuda", dtype=torch.bfloat16)
    Bt[:, 8:8 + N] = B.t()
    a = At[:, 8:8 + M] if a_mn else A
    b = Bt[:, 8:8 + N] if b_mn else B
    # plain GEMM
    ref = ops.gemm_bf16_tn(A, B)
    out = ops.gemm_bf16_tn(a, b, a_mn=a_mn, b_mn=b_mn)
    torch.cuda.synchronize()
    assert torch.equal(ref, out)
    f32 = A.float() @ B.float().t()
    assert ((out - f32).abs().max() / f32.abs().max()).item() < 1e-4
    # accumulating (split-K) GEMM: reduce-add order is not deterministic, compare numerically
    acc = torch.zeros(M, N, device="cuda")
    ops.gemm_bf16_tn(a, b, out=acc, accumulate=True, a_mn=a_mn, b_mn=b_mn)
    torch.cuda.synchronize()
    assert ((acc - f32).abs().max() / f32.abs().max()).item() < 1e-4
