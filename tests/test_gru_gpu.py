"""GPU parity: persistent GRU kernels (through the C ABI) vs torch.nn.GRU in fp32/fp64 on CPU.

The kernels use bf16 tensor-core operands with fp32 accumulation and fp32 gate math, so the
tolerance is the bf16 operand rounding (2^-9 relative per product), not fp32 epsilon:
outputs within 2e-2 absolute of the fp64 reference (|h| <= 1), gradients within 3% of the
largest reference gradient entry.
"""
import pytest
import torch

pytestmark = pytest.mark.gpu


def _ref_and_ours(B, T, In, H, L, bidir, seed):
    from speech_b200.ops import gru_stack
    torch.manual_seed(seed)
    rnn = torch.nn.GRU(In, H, L, batch_first=True, bidirectional=bidir)
    x = torch.randn(B, T, In)
    # fp64 CPU reference
    rnn64 = torch.nn.GRU(In, H, L, batch_first=True, bidirectional=bidir).double()
    rnn64.load_state_dict({k: v.double() for k, v in rnn.state_dict().items()})
    x64 = x.double().requires_grad_(True)
    y64, _ = rnn64(x64)
    w = torch.randn_like(y64)
    (y64 * w).sum().backward()
    # ours
    rnn_c = rnn.cuda()
    xc = x.cuda().requires_grad_(True)
    yc = gru_stack(xc, rnn_c)
    (yc * w.float().cuda()).sum().backward()
    torch.cuda.synchronize()
    return rnn64, x64, y64, rnn_c, xc, yc


@pytest.mark.parametrize("B,T,In,H,L,bidir", [
    (4, 12, 160, 16, 1, False),    # tests/shared.py tiny config (uni, dim 16)
    (3, 9, 40, 32, 2, True),       # ragged batch (padded to 8), 2 layers bi
    (8, 20, 64, 128, 2, True),     # several CTAs per direction
    (16, 31, 480, 256, 3, True),   # shipped-config width
    # uni H = 1280: the backward K split would need 5 chunk groups of its 4 full barriers, so the
    # backward must take the full gather at 8 and 16 rows, where kt / ks would otherwise be picked
    (8, 5, 64, 1280, 1, False),
    (16, 5, 64, 1280, 1, False),
])
def test_gru_stack_forward_backward(cuda_lib, B, T, In, H, L, bidir):
    rnn64, x64, y64, rnn_c, xc, yc = _ref_and_ours(B, T, In, H, L, bidir, seed=B + T + H)
    err = (yc.double().cpu() - y64).abs().max().item()
    assert err < 2e-2, err
    gx = xc.grad.double().cpu()
    assert (gx - x64.grad).abs().max().item() < 3e-2 * x64.grad.abs().max().item() + 1e-4
    for (n, p64), (_, pc) in zip(rnn64.named_parameters(), rnn_c.named_parameters()):
        g = pc.grad.double().cpu()
        ref = p64.grad
        tol = 3e-2 * ref.abs().max().item() + 1e-4
        assert (g - ref).abs().max().item() < tol, n


def test_gru_north_star_width_short(cuda_lib):
    """H=1024 (64 CTAs per direction, both directions resident), B=64, short T."""
    rnn64, x64, y64, rnn_c, xc, yc = _ref_and_ours(64, 6, 480, 1024, 1, True, seed=5)
    assert (yc.double().cpu() - y64).abs().max().item() < 2e-2
    for (n, p64), (_, pc) in zip(rnn64.named_parameters(), rnn_c.named_parameters()):
        ref = p64.grad
        assert (pc.grad.double().cpu() - ref).abs().max().item() < 3e-2 * ref.abs().max().item() + 1e-4, n


@pytest.mark.parametrize("B", [8, 16, 32])
def test_gru_north_star_width_small_batches(cuda_lib, B):
    """per-rank batches of the 8/4/2-GPU strong-scaling runs (64/N) at H=1024."""
    rnn64, x64, y64, rnn_c, xc, yc = _ref_and_ours(B, 5, 480, 1024, 1, True, seed=B)
    assert (yc.double().cpu() - y64).abs().max().item() < 2e-2
    for (n, p64), (_, pc) in zip(rnn64.named_parameters(), rnn_c.named_parameters()):
        ref = p64.grad
        assert (pc.grad.double().cpu() - ref).abs().max().item() < 3e-2 * ref.abs().max().item() + 1e-4, n


@pytest.mark.parametrize("B,H", [(96, 256), (128, 256), (128, 1024)])
def test_gru_large_per_gpu_batch(cuda_lib, B, H):
    """batches above 64 rows per GPU (all four TMEM lane quadrants; smaller smem ring at H=1024)."""
    rnn64, x64, y64, rnn_c, xc, yc = _ref_and_ours(B, 4, 64, H, 1, True, seed=B + H)
    assert (yc.double().cpu() - y64).abs().max().item() < 2e-2
    for (n, p64), (_, pc) in zip(rnn64.named_parameters(), rnn_c.named_parameters()):
        ref = p64.grad
        assert (pc.grad.double().cpu() - ref).abs().max().item() < 3e-2 * ref.abs().max().item() + 1e-4, n


@pytest.mark.parametrize("B", [8, 20, 33, 56, 64])
def test_gru_both_k_split_flavours(cuda_lib, B):
    """The two K-split recurrence kernels (batch-major accumulator `ks`, transposed accumulator
    `kt`), forward and backward.  csrc/gru.cu picks the flavour by padded batch size; 8/24/40/56/64
    rows reach every kernel the selection can pick: forward `kt<1>` at 8, `kt<2>` at 24, `ks` at
    40-64; backward `kt<1>` at 8, `ks` at 24-64."""
    rnn64, x64, y64, rnn_c, xc, yc = _ref_and_ours(B, 7, 96, 256, 2, True, seed=B)
    assert (yc.double().cpu() - y64).abs().max().item() < 2e-2
    gx = xc.grad.double().cpu()
    assert (gx - x64.grad).abs().max().item() < 3e-2 * x64.grad.abs().max().item() + 1e-4
    for (n, p64), (_, pc) in zip(rnn64.named_parameters(), rnn_c.named_parameters()):
        ref = p64.grad
        assert (pc.grad.double().cpu() - ref).abs().max().item() < 3e-2 * ref.abs().max().item() + 1e-4, n


def test_gru_wgrad_accumulates_into_existing_grad(cuda_lib):
    """With .grad already allocated (FlatSGD / zero_grad(set_to_none=False)) the weight-gradient
    GEMMs reduce-add straight into it; two backward passes must give exactly 2x one pass."""
    from speech_b200 import ops
    from speech_b200.ops import gru_stack
    torch.manual_seed(3)
    rnn = torch.nn.GRU(64, 128, 2, batch_first=True, bidirectional=True).cuda()
    x = torch.randn(8, 7, 64).cuda()
    gru_stack(x, rnn).sum().backward()                    # .grad is None -> returned-gradient path
    ref = [p.grad.clone() for p in rnn.parameters()]
    for p in rnn.parameters():
        p.grad.zero_()
    ops.set_grad_sink(True)                               # what optim.FlatSGD switches on
    gru_stack(x, rnn).sum().backward()                    # fused accumulation path
    for p, r in zip(rnn.parameters(), ref):
        assert torch.allclose(p.grad, r, rtol=1e-5, atol=1e-6)
    gru_stack(x, rnn).sum().backward()
    for p, r in zip(rnn.parameters(), ref):
        assert torch.allclose(p.grad, 2 * r, rtol=1e-5, atol=1e-6)


def test_gru_minibatch_above_one_launch_is_chunked(cuda_lib):
    """A minibatch of more rows than one recurrence launch holds (128) runs as consecutive chunks;
    utterances are independent, so outputs and gradients still match the fp64 reference."""
    rnn64, x64, y64, rnn_c, xc, yc = _ref_and_ours(150, 5, 32, 64, 2, True, seed=150)
    assert yc.shape == y64.shape
    assert (yc.double().cpu() - y64).abs().max().item() < 2e-2
    assert (xc.grad.double().cpu() - x64.grad).abs().max().item() < \
        3e-2 * x64.grad.abs().max().item() + 1e-4
    for (n, p64), (_, pc) in zip(rnn64.named_parameters(), rnn_c.named_parameters()):
        ref = p64.grad
        assert (pc.grad.double().cpu() - ref).abs().max().item() < 3e-2 * ref.abs().max().item() + 1e-4, n


def test_gru_default_path_returns_gradients_to_autograd(cuda_lib):
    """Without the FlatSGD opt-in the Function has no side effect on .grad: torch.autograd.grad
    gets every weight gradient even when .grad buffers already exist, and leaves them untouched."""
    from speech_b200.ops import gru_stack
    torch.manual_seed(4)
    rnn = torch.nn.GRU(32, 64, 2, batch_first=True, bidirectional=True).cuda()
    x = torch.randn(5, 6, 32).cuda()
    gru_stack(x, rnn).sum().backward()
    want = [p.grad.clone() for p in rnn.parameters()]
    for p in rnn.parameters():
        p.grad.fill_(7.0)
    got = torch.autograd.grad(gru_stack(x, rnn).sum(), list(rnn.parameters()))
    for g, w, p in zip(got, want, rnn.parameters()):
        assert g is not None and torch.allclose(g, w, rtol=1e-5, atol=1e-6)
        assert torch.all(p.grad == 7.0)


@pytest.mark.parametrize("B,T,In,H,L", [(6, 11, 40, 32, 3), (8, 9, 64, 128, 2)])
def test_gru_inter_layer_dropout_matches_masked_reference(cuda_lib, B, T, In, H, L):
    """nn.GRU(dropout=p) semantics in training: every layer output but the last is multiplied by
    a keep mask / (1-p).  The masks are drawn with torch.rand on the device in layer order over
    the kernels' time-major padded layout (row t*Bp + b), so re-seeding reproduces them for an
    fp64 layer-by-layer reference; forward and all gradients must match (bf16 operand bars)."""
    from speech_b200.ops import gru_stack
    p = 0.3
    torch.manual_seed(B + T)
    rnn = torch.nn.GRU(In, H, L, batch_first=True, bidirectional=True, dropout=p).cuda()
    x = torch.randn(B, T, In).cuda().requires_grad_(True)
    torch.manual_seed(1234)
    y = gru_stack(x, rnn, dropout=p)
    assert y.dtype == torch.float32
    w = torch.randn_like(y)
    (y * w).sum().backward()
    got = {n: q.grad.double().cpu() for n, q in rnn.named_parameters()}
    # ---- reference: one fp64 nn.GRU per layer, same masks ----
    Bp = (B + 7) // 8 * 8
    torch.manual_seed(1234)
    masks = [(torch.rand(T * Bp, 2 * H, device="cuda") >= p).double().cpu() / (1.0 - p)
             for _ in range(L - 1)]
    h = x.detach().double().cpu().requires_grad_(True)
    x64 = h
    layers = []
    for l in range(L):
        g = torch.nn.GRU(In if l == 0 else 2 * H, H, 1, batch_first=True, bidirectional=True).double()
        sd = {}
        for k, v in rnn.state_dict().items():
            if "_l%d" % l in k:
                sd[k.replace("_l%d" % l, "_l0")] = v.double().cpu()
        g.load_state_dict(sd)
        layers.append(g)
        h, _ = g(h)
        if l + 1 < L:
            mk = masks[l].view(T, Bp, 2 * H)[:, :B].transpose(0, 1)
            h = h * mk
    (h * w.double().cpu()).sum().backward()
    assert (y.double().cpu() - h.detach()).abs().max().item() < 3e-2
    assert (x.grad.double().cpu() - x64.grad).abs().max().item() < \
        3e-2 * x64.grad.abs().max().item() + 1e-4
    for l, g in enumerate(layers):
        for k, q in g.named_parameters():
            name = k.replace("_l0", "_l%d" % l)
            ref = q.grad
            assert (got[name] - ref).abs().max().item() < 3e-2 * ref.abs().max().item() + 1e-4, name
    # dropout really happened, and eval (dropout=0) is deterministic and different
    y0 = gru_stack(x.detach(), rnn, dropout=0.0)
    assert not torch.allclose(y0, y.detach(), atol=1e-3)
