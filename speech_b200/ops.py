"""Host-side operators over the C ABI: dense contraction and the (bi)GRU stack.

PyTorch is used here for device memory, streams and autograd plumbing only; the arithmetic of
the recurrence and of every projection runs in the hand-written sm_100a kernels of csrc/.
Internal activations are TIME-MAJOR with the batch padded to a multiple of 8 (row m = t*Bp + b).
"""
import ctypes

import torch

from . import _lib

GEMM_ACCUMULATE = 1
GEMM_ROW_REMAP = 2
GEMM_A_MN = 4
GEMM_B_MN = 8


def _round_up(x, m):
    return (x + m - 1) // m * m


# ---- optional per-kernel timing (CUDA events on the launching stream; used by bench.py) ----
_prof = None
_prof_detail = False      # developer: one profile class per GEMM shape (tools/debug_step.py)


def profile_begin():
    global _prof
    _prof = []


def profile_end():
    """-> {kernel class: (launches, total ms, total algorithmic FLOPs)}"""
    global _prof
    rec, _prof = _prof, None
    torch.cuda.synchronize()
    out = {}
    for name, flops, e0, e1 in rec or []:
        n, ms, fl = out.get(name, (0, 0.0, 0.0))
        out[name] = (n + 1, ms + e0.elapsed_time(e1), fl + flops)
    return out


def _launch(name, flops, fn):
    """Run one C-ABI launch; counts it and, when profiling, brackets it with CUDA events."""
    _lib.launch_count += 1
    if _prof is None:
        return _lib.check(fn(), name)
    e0 = torch.cuda.Event(enable_timing=True)
    e1 = torch.cuda.Event(enable_timing=True)
    e0.record()
    rc = fn()
    e1.record()
    _prof.append((name, flops, e0, e1))
    return _lib.check(rc, name)


def gemm_bf16_tn(A, B, out=None, bias=None, accumulate=False, split_k=1, remap=None,
                 a_mn=False, b_mn=False):
    """out[M,N] (f32) (+)= A[M,K] (bf16) @ B[N,K]^T (bf16) (+ bias).  A/B may be row-strided views.

    a_mn / b_mn: that operand is given as [K][M] / [K][N] (the contraction runs over its rows).
    remap=(Bp, T, valid_B): rows m = t*Bp + b are written batch-first to row b*T + t.
    """
    lib = _lib.load()
    assert A.dtype == torch.bfloat16 and B.dtype == torch.bfloat16
    assert A.stride(1) == 1 and B.stride(1) == 1
    K, M = A.shape if a_mn else (A.shape[1], A.shape[0])
    Kb, N = B.shape if b_mn else (B.shape[1], B.shape[0])
    assert K == Kb
    flags = (GEMM_A_MN if a_mn else 0) | (GEMM_B_MN if b_mn else 0)
    rB = rT = vB = 0
    if remap is not None:
        rB, rT, vB = remap
        flags |= GEMM_ROW_REMAP
        rows = vB * rT
    else:
        rows = M
    if out is None:
        assert not accumulate
        out = torch.empty(rows, N, dtype=torch.float32, device=A.device)
    assert out.dtype == torch.float32 and out.stride(1) == 1 and out.shape[0] >= rows
    if accumulate:
        flags |= GEMM_ACCUMULATE
    sp = _lib.stream_ptr()
    name = "gemm_bf16_tn"
    if _prof_detail:
        name = "gemm %dx%dx%d%s%s%s" % (M, N, K, " aT" if a_mn else "", " bT" if b_mn else "",
                                       " acc" if accumulate else "")
    _launch(name, 2.0 * M * N * K,
            lambda: lib.sb_gemm_bf16_tn(A.data_ptr(), A.stride(0), B.data_ptr(), B.stride(0),
                                        out.data_ptr(), out.stride(0), _lib.ptr(bias), M, N, K,
                                        flags, split_k, rB, rT, vB, sp))
    return out


# ------------------------------------------------------------------------------------------------
# "Parity mode" (SURVEY.md section 7): the forward pass of the encoder in reference precision, to
# measure the bf16 tensor-core path against.  Dense contractions run as 3-pass split-bf16 GEMMs
# (x = hi + lo with hi = bf16(x), lo = bf16(x - hi): hi*hi + hi*lo + lo*hi on the tensor cores,
# relative error ~2^-16), the recurrence in plain fp32 (csrc/gru_f32.cu).  No autograd.
# ------------------------------------------------------------------------------------------------
def _split_bf16(t, Kp):
    t = t.detach().float()
    hi = t.to(torch.bfloat16)
    lo = (t - hi.float()).to(torch.bfloat16)
    if Kp != t.shape[1]:
        hi = torch.nn.functional.pad(hi, (0, Kp - t.shape[1]))
        lo = torch.nn.functional.pad(lo, (0, Kp - t.shape[1]))
    return hi.contiguous(), lo.contiguous()


def gemm_split(A, B, bias=None, remap=None):
    """A (M,K) f32 @ B (N,K)^T f32 -> (M,N) f32 with split-bf16 operands (3 tensor-core passes)."""
    Kp = _round_up(A.shape[1], 8)
    a_hi, a_lo = _split_bf16(A, Kp)
    b_hi, b_lo = _split_bf16(B, Kp)
    out = gemm_bf16_tn(a_hi, b_hi, bias=bias, remap=remap)
    gemm_bf16_tn(a_hi, b_lo, out=out, accumulate=True, remap=remap)
    gemm_bf16_tn(a_lo, b_hi, out=out, accumulate=True, remap=remap)
    return out


def encode_logits_parity(x, conv, rnn, fc):
    """Reference-precision forward of conv stack -> GRU stack -> halves-sum -> fc (no grad):
    x (B,T,F) -> logits (B,T',V).  Same kernels' layouts, split-bf16 GEMMs, fp32 recurrence."""
    _lib.require_cuda(x, "x")
    lib = _lib.load()
    dev = x.device
    B, Ti, Fi = x.shape
    sp = _lib.stream_ptr()
    cur = x.detach().float().contiguous()              # (B, Ti, Fi, Ci) channels-last, Ci = 1
    Ci = 1
    for l, c in enumerate(m for m in conv.children() if isinstance(m, torch.nn.Conv2d)):
        kh, kw, s_ = c.kernel_size[0], c.kernel_size[1], c.stride[0]
        Co = c.out_channels
        K = kh * kw * Ci
        Kp = _round_up(K, 8)
        To, Fo = (Ti - kh) // s_ + 1, (Fi - kw) // s_ + 1
        M = B * To * Fo
        r = cur if l == 0 else torch.relu(cur)
        r_hi = r.to(torch.bfloat16).float()
        parts = []
        for src in (r_hi, r - r_hi):                   # im2col of the hi and lo halves (exact)
            A = torch.empty(M, Kp, dtype=torch.bfloat16, device=dev)
            _launch("conv_im2col", 0.0,
                    lambda: lib.sb_conv_im2col(src.data_ptr(), None, 1.0, A.data_ptr(), B, Ti, Fi,
                                               Ci, kh, kw, s_, Kp, 0, sp))
            parts.append(A)
        W = torch.zeros(Co, Kp, dtype=torch.float32, device=dev)
        W[:, :K] = c.weight.detach().float().permute(0, 2, 3, 1).reshape(Co, K)
        w_hi, w_lo = _split_bf16(W, Kp)
        C = gemm_bf16_tn(parts[0], w_hi, bias=c.bias.detach().float().contiguous())
        gemm_bf16_tn(parts[0], w_lo, out=C, accumulate=True)
        gemm_bf16_tn(parts[1], w_hi, out=C, accumulate=True)
        cur, Ti, Fi, Ci = C, To, Fo, Co
    feats = torch.empty(B, Ti, Ci * Fi, dtype=torch.float32, device=dev)
    _launch("conv_relu_to_bct", 0.0,
            lambda: lib.sb_conv_relu_to_bct(cur.data_ptr(), None, 1.0, feats.data_ptr(), B, Ti, Fi,
                                            Ci, sp))
    ndir, weights = _gru_weights(rnn)
    H = rnn.hidden_size
    T = Ti
    Bp = _round_up(B, 8)
    M = T * Bp
    X = torch.zeros(T, Bp, feats.shape[2], dtype=torch.float32, device=dev)
    X[:, :B] = feats.transpose(0, 1)
    X = X.view(M, -1)
    barrier = torch.zeros(2, dtype=torch.int32, device=dev)
    for l in range(rnn.num_layers):
        wl = weights[l * 4 * ndir:(l + 1) * 4 * ndir]
        w_ih = torch.cat([wl[d * 4].detach().float() for d in range(ndir)])
        b_ih = torch.cat([wl[d * 4 + 2].detach().float() for d in range(ndir)]).contiguous()
        w_hh = torch.stack([wl[d * 4 + 1].detach().float() for d in range(ndir)]).contiguous()
        b_hh = torch.stack([wl[d * 4 + 3].detach().float() for d in range(ndir)]).contiguous()
        gi = gemm_split(X, w_ih, bias=b_ih)
        y = torch.empty(M, ndir * H, dtype=torch.float32, device=dev)
        _launch("gru_fwd_f32", 2.0 * M * 3 * H * H * ndir,
                lambda: lib.sb_gru_fwd_f32(gi.data_ptr(), w_hh.data_ptr(), b_hh.data_ptr(),
                                           y.data_ptr(), barrier.data_ptr(), T, Bp, H, ndir, sp))
        X = y
    w = fc.weight.detach().float()
    wcat = torch.cat([w, w], 1) if ndir == 2 else w
    V = w.shape[0]
    return gemm_split(X, wcat, bias=fc.bias.detach().float().contiguous(),
                      remap=(Bp, T, B)).view(B, T, V)


class LinearFunction(torch.autograd.Function):
    """y = x W^T + b on the tcgen05 GEMM (bf16 operands, fp32 accumulate), forward and backward:
    the arithmetic behind the reference's LinearND / nn.Linear (model.py:115-133).
    x (N, K) f32, W (O, K), b (O) -> (N, O) f32."""

    @staticmethod
    def forward(ctx, x, w, b):
        _lib.require_cuda(x, "x")
        N, K = x.shape
        Kp = _round_up(K, 8)
        xb = x.detach().to(torch.bfloat16)
        wb = w.detach().to(torch.bfloat16)
        if Kp != K:
            xb = torch.nn.functional.pad(xb, (0, Kp - K))
            wb = torch.nn.functional.pad(wb, (0, Kp - K))
        xb, wb = xb.contiguous(), wb.contiguous()
        ctx.save_for_backward(xb, wb)
        ctx.K = K
        ctx.has_bias = b is not None
        return gemm_bf16_tn(xb, wb, bias=None if b is None else b.detach().float().contiguous())

    @staticmethod
    def backward(ctx, dy):
        xb, wb = ctx.saved_tensors
        K = ctx.K
        O = wb.shape[0]
        Op = _round_up(O, 8)
        dyb = dy.detach().to(torch.bfloat16)
        if Op != O:
            dyb = torch.nn.functional.pad(dyb, (0, Op - O))
            wb = torch.nn.functional.pad(wb, (0, 0, 0, Op - O))
        dyb, wb = dyb.contiguous(), wb.contiguous()
        dx = dw = db = None
        if ctx.needs_input_grad[0]:
            dx = gemm_bf16_tn(dyb, wb, b_mn=True)[:, :K]          # dY W: W is the [K][N] form
        if ctx.needs_input_grad[1]:
            dw = torch.zeros(Op, xb.shape[1], dtype=torch.float32, device=dy.device)
            gemm_bf16_tn(dyb, xb, out=dw, accumulate=True, a_mn=True, b_mn=True)   # dY^T X
            dw = dw[:O, :K]
        if ctx.has_bias and ctx.needs_input_grad[2]:
            db = dy.sum(0)
        return dx, dw, db


def linear(x, w, b=None):
    """nn.Linear semantics over the last dimension of an N-D CUDA tensor, on the tcgen05 GEMM."""
    lead = x.shape[:-1]
    out = LinearFunction.apply(x.reshape(-1, x.shape[-1]).float(), w, b)
    return out.view(*lead, out.shape[-1])


_gru_operands = {}


def register_gru_operands(first_w_ih, entry):
    """optim.FlatSGD: operands of one GRU layer as views of its flat buffers (see there)."""
    _gru_operands[id(first_w_ih)] = entry


def _cached_gru_operands(w_ih0, Kl):
    e = _gru_operands.get(id(w_ih0))
    if e is None or e["wih"].shape[1] != Kl or e["params"][0] is not w_ih0:
        return None
    if any(q._version != v for q, v in zip(e["params"], e["versions"])):
        return None          # modified outside FlatSGD.step(): fall back to casting the fp32 values
    return e


_grad_ready_hook = None
_announce = True
_grad_sink_enabled = False


def set_grad_sink(enabled):
    """Opt-in (optim.FlatSGD): let the weight-gradient GEMMs of GRUStackFunction.backward
    accumulate straight into the parameters' existing .grad buffers and return None to autograd
    for them.  Off by default, so that torch.autograd.grad, gradcheck, tensor hooks and gradient
    accumulation see ordinary returned gradients."""
    global _grad_sink_enabled
    _grad_sink_enabled = bool(enabled)


_grad_guard = None


def set_grad_ready_hook(fn, guard=None):
    """fn(list_of_parameters) is called from inside GRUStackFunction.backward as soon as the
    gradients of one layer's parameters are final in their .grad buffers (all producing kernels
    enqueued on the current stream).  Used by optim.FlatSGD to start that layer's all-reduce
    while the layers below are still being differentiated.  None disables.
    guard(parameters) (optional) runs at the START of every announcing backward of a GRU stack,
    before any gradient buffer is touched: it raises if gradients of these parameters were
    already announced in this step (a second backward pass would add local gradients into
    slices that are being all-reduced)."""
    global _grad_ready_hook, _grad_guard
    _grad_ready_hook = fn
    _grad_guard = guard if fn is not None else None


def _bias_sink(param):
    if not _grad_sink_enabled:
        return None
    g = getattr(param, "grad", None)
    if g is None or not g.is_cuda or g.dtype != torch.float32:
        return None
    return g


def _grad_sink(param, rows=None):
    """The parameter's existing .grad (optionally a row slice) if the weight-gradient GEMM can
    accumulate straight into it (fp32, contiguous, 16-byte aligned rows), else None.  Writing
    dW with the GEMM's reduce-add epilogue into .grad replaces a zero-filled temporary plus
    autograd's separate `grad += dW` pass (the gradient-accumulation fusion used by large-model
    trainers); the Function then returns None for that parameter."""
    if not _grad_sink_enabled:
        return None
    g = getattr(param, "grad", None)
    if g is None or not g.is_cuda or g.dtype != torch.float32 or not g.is_contiguous():
        return None
    if g.dim() != 2 or (g.stride(0) % 4) != 0 or (g.data_ptr() % 16) != 0:
        return None
    return g if rows is None else g[rows[0]:rows[1]]


def _workspace(nbytes, dev):
    """1024-byte aligned scratch for one recurrence launch (counters + exchange tiles)"""
    buf = torch.empty(nbytes + 1024, dtype=torch.uint8, device=dev)
    off = (-buf.data_ptr()) % 1024
    return buf[off:off + nbytes]


class GRUStackFunction(torch.autograd.Function):
    """Multi-layer (bi)directional GRU, semantics of nn.GRU(batch_first=True) with h0 = 0.

    forward(x (B,T,In) f32 cuda, ndir, H, train, *weights) -> (B,T,ndir*H) f32
    weights: per layer, per direction: w_ih (3H,In_l), w_hh (3H,H), b_ih (3H), b_hh (3H)
    (the parameter order of nn.GRU: weight_ih_l{k}[_reverse], weight_hh_..., bias_ih_..., bias_hh_...)
    """

    @staticmethod
    def forward(ctx, x, ndir, H, dropout, fc_w, fc_b, *weights):
        """fc_w/fc_b (optional): fuse `LinearND(sum of direction halves)` (reference
        model.py:75-77 + ctc_model.py:29) as ONE contraction on the bf16 top-layer output:
        (h_f + h_b) W^T = [h_f | h_b] [W | W]^T, written batch-first by the GEMM epilogue."""
        _lib.require_cuda(x, "x")
        lib = _lib.load()
        B, T, In = x.shape
        dev = x.device
        L = len(weights) // (4 * ndir)
        Bp = _round_up(B, 8)
        if Bp > 128:
            raise _lib.SpeechB200Error("per-GPU batch > 128 not supported by the GRU kernel yet")
        M = T * Bp
        D = ndir * H
        need_grad = any(ctx.needs_input_grad)     # all False under torch.no_grad()

        # layer-0 operand: time-major, batch padded, K padded to a multiple of 8, bf16
        Inp = _round_up(In, 8)
        if B == Bp and In == Inp:
            X = x.detach().transpose(0, 1).to(torch.bfloat16).reshape(M, Inp)
        else:
            X = torch.zeros(T, Bp, Inp, dtype=torch.bfloat16, device=dev)
            X[:, :B, :In] = x.transpose(0, 1)
            X = X.view(M, Inp)
        nbytes = ctypes.c_size_t(0)
        _lib.check(lib.sb_gru_fwd_workspace_size(Bp, H, ndir, ctypes.byref(nbytes)), "ws")
        ws = _workspace(nbytes.value, dev)
        saved = []
        y = None
        for l in range(L):
            wl = weights[l * 4 * ndir:(l + 1) * 4 * ndir]
            w_ih = [wl[d * 4 + 0] for d in range(ndir)]
            w_hh = [wl[d * 4 + 1] for d in range(ndir)]
            b_ih = [wl[d * 4 + 2] for d in range(ndir)]
            b_hh = [wl[d * 4 + 3] for d in range(ndir)]
            Kl = X.shape[1]
            In_l = w_ih[0].shape[1]
            cached = _cached_gru_operands(w_ih[0], Kl)
            if cached is not None:
                # views of the optimizer's flat buffers (bf16 shadow written by sgd_clip_step)
                wih_cat, whh = cached["wih"], cached["whh"]
                bih_cat, bhh = cached["bih"], cached["bhh"]
            else:
                # bf16 operand copies of the master weights: one fused cast+copy per matrix
                wih_cat = (torch.empty if Kl == In_l else torch.zeros)(
                    ndir * 3 * H, Kl, dtype=torch.bfloat16, device=dev)
                whh = torch.empty(ndir, 3 * H, H, dtype=torch.bfloat16, device=dev)
                for d in range(ndir):
                    wih_cat[d * 3 * H:(d + 1) * 3 * H, :In_l].copy_(w_ih[d].detach())
                    whh[d].copy_(w_hh[d].detach())
                bih_cat = torch.cat([b.detach() for b in b_ih]).float().contiguous()
                bhh = torch.stack([b.detach() for b in b_hh]).float().contiguous()
            gi = gemm_bf16_tn(X, wih_cat, bias=bih_cat)
            y = torch.empty(M, D, dtype=torch.float32, device=dev)
            xn = torch.empty(M, D, dtype=torch.bfloat16, device=dev)
            gates = None
            if need_grad:
                gates = torch.empty(M, ndir, 4, H, dtype=torch.float32, device=dev)
            sp = _lib.stream_ptr()
            _launch("gru_fwd", 2.0 * M * 3 * H * H * ndir,
                    lambda: lib.sb_gru_fwd(gi.data_ptr(), whh.data_ptr(), bhh.data_ptr(),
                                           y.data_ptr(), xn.data_ptr(), _lib.ptr(gates),
                                           ws.data_ptr(), nbytes.value, T, Bp, H, ndir, sp))
            mask = None
            hb = xn                                     # bf16 h_t (un-masked): dW_hh operand
            if dropout > 0.0 and l + 1 < L:
                # inter-layer dropout of nn.GRU(dropout=p): applied to every layer output but the last
                mask = (torch.rand(M, D, device=dev) >= dropout).float() * (1.0 / (1.0 - dropout))
                # the next layer's operand stays bf16 (bf16 * f32 would promote to f32): mask the
                # fp32 state and round once
                xn = (y * mask).to(torch.bfloat16)
            if need_grad:
                saved.append((X, y, gates, mask, wih_cat, whh, hb))
            X = xn
        ctx.saved = saved
        ctx.announce = _announce
        ctx.weights = weights
        ctx.dims = (B, T, In, Bp, H, ndir, L)
        ctx.fc = None
        if fc_w is not None:
            V = fc_w.shape[0]
            wcat = fc_w.detach().to(torch.bfloat16)
            if ndir == 2:
                wcat = torch.cat([wcat, wcat], 1)
            wcat = wcat.contiguous()
            out = gemm_bf16_tn(X, wcat, bias=fc_b.detach().float().contiguous(),
                               remap=(Bp, T, B)).view(B, T, V)
            ctx.fc = (fc_w, X)
            return out
        out = y.view(T, Bp, D)[:, :B].transpose(0, 1).contiguous()
        return out

    @staticmethod
    def backward(ctx, dout):
        lib = _lib.load()
        B, T, In, Bp, H, ndir, L = ctx.dims
        weights = ctx.weights
        if _grad_ready_hook is not None and ctx.announce and _grad_guard is not None:
            _grad_guard(list(weights))
        dev = dout.device
        M = T * Bp
        D = ndir * H
        K3 = 3 * H
        dfc_w = dfc_b = None
        if ctx.fc is not None:
            fc_w, Xtop = ctx.fc
            V = fc_w.shape[0]
            Vp = _round_up(V, 8)
            dl = torch.zeros(T, Bp, Vp, dtype=torch.bfloat16, device=dev)
            dl[:, :B, :V] = dout.transpose(0, 1)
            dl = dl.view(M, Vp)
            w = fc_w.detach().to(torch.bfloat16)
            wT = torch.zeros(D, Vp, dtype=torch.bfloat16, device=dev)      # [D][Vp] = [W | W]^T
            for d in range(ndir):
                wT[d * H:(d + 1) * H, :V] = w.t()
            dY = gemm_bf16_tn(dl, wT)                                         # [M][D] f32
            dw2 = torch.zeros(Vp, D, dtype=torch.float32, device=dev)
            # dW (Vp x D) = dl^T Xtop, both operands read token-major (MN-major UMMA)
            gemm_bf16_tn(dl, Xtop, out=dw2, accumulate=True, a_mn=True, b_mn=True)
            dfc_w = dw2[:V, :H] if ndir == 1 else dw2[:V, :H] + dw2[:V, H:]
            dfc_b = dout.sum((0, 1))
        elif B == Bp:
            # (dout may be an expanded stride-0 tensor, e.g. from y.sum(): force a real copy)
            dY = dout.transpose(0, 1).float().contiguous().view(M, D)
        else:
            dY = torch.zeros(T, Bp, D, dtype=torch.float32, device=dev)
            dY[:, :B] = dout.transpose(0, 1)
            dY = dY.view(M, D)
        nbytes = ctypes.c_size_t(0)
        _lib.check(lib.sb_gru_bwd_workspace_size(Bp, H, ndir, ctypes.byref(nbytes)), "ws")
        ws = _workspace(nbytes.value, dev)
        grads = [None] * len(weights)
        for l in reversed(range(L)):
            X, y, gates, mask, wih_cat, whh, hb = ctx.saved[l]
            if mask is not None:
                dY = dY * mask
            wl = weights[l * 4 * ndir:(l + 1) * 4 * ndir]
            Kl = X.shape[1]
            In_l = wl[0].shape[1]
            dgi = torch.empty(M, ndir * K3, dtype=torch.bfloat16, device=dev)
            dghn = torch.empty(M, D, dtype=torch.bfloat16, device=dev)
            dbih = torch.zeros(ndir * K3, dtype=torch.float32, device=dev)
            dbhh = torch.zeros(ndir * K3, dtype=torch.float32, device=dev)
            sp = _lib.stream_ptr()
            _launch("gru_bwd", 2.0 * M * 3 * H * H * ndir,
                    lambda dY=dY: lib.sb_gru_bwd(dY.data_ptr(), y.data_ptr(), gates.data_ptr(),
                                                 whh.data_ptr(), dgi.data_ptr(), dghn.data_ptr(),
                                                 dbih.data_ptr(), dbhh.data_ptr(), ws.data_ptr(),
                                                 nbytes.value, T, Bp, H, ndir, sp))
            base = l * 4 * ndir
            # ---- weight gradients: contract the token-major operands over their rows ----
            Ms = M - Bp                      # tokens that have a predecessor in the recurrence
            for d in range(ndir):
                # dW_ih[d] (3H x In_l) = dgi[:, d]^T X
                sink = _grad_sink(wl[d * 4])
                dwih = sink if sink is not None else \
                    torch.zeros(K3, In_l, dtype=torch.float32, device=dev)
                gemm_bf16_tn(dgi[:, d * K3:(d + 1) * K3], X[:, :In_l], out=dwih,
                             accumulate=True, a_mn=True, b_mn=True)
                # dW_hh[d] = [dgi_r | dgi_z | dghn]^T h_prev: h_prev of token (t, b) is token
                # (t-1, b) in the forward direction and (t+1, b) in the reverse one, so the
                # shift is a row offset of Bp on one of the two operands
                sink_hh = _grad_sink(wl[d * 4 + 1])
                dwhh = sink_hh if sink_hh is not None else \
                    torch.zeros(K3, H, dtype=torch.float32, device=dev)
                if Ms > 0:
                    ga, hp = (slice(Bp, M), slice(0, Ms)) if d == 0 else \
                        (slice(0, Ms), slice(Bp, M))
                    gemm_bf16_tn(dgi[ga, d * K3:d * K3 + 2 * H], hb[hp, d * H:(d + 1) * H],
                                 out=dwhh[:2 * H], accumulate=True, a_mn=True, b_mn=True)
                    gemm_bf16_tn(dghn[ga, d * H:(d + 1) * H], hb[hp, d * H:(d + 1) * H],
                                 out=dwhh[2 * H:], accumulate=True, a_mn=True, b_mn=True)
                grads[base + d * 4 + 0] = None if sink is not None else dwih
                grads[base + d * 4 + 1] = None if sink_hh is not None else dwhh
                grads[base + d * 4 + 2] = dbih[d * K3:(d + 1) * K3]
                grads[base + d * 4 + 3] = dbhh[d * K3:(d + 1) * K3]
            if _grad_ready_hook is not None and ctx.announce:
                base = l * 4 * ndir
                if all(grads[base + d * 4 + k] is None for d in range(ndir) for k in (0, 1)):
                    # weights already sit in .grad; add the biases there too, then announce
                    ok = True
                    for d in range(ndir):
                        for k in (2, 3):
                            sink = _bias_sink(wl[d * 4 + k])
                            if sink is None:
                                ok = False
                                continue
                            sink.add_(grads[base + d * 4 + k])
                            grads[base + d * 4 + k] = None
                    if ok:
                        _grad_ready_hook(list(wl))
            # ---- gradient w.r.t. the layer input ----
            if l > 0 or ctx.needs_input_grad[0]:
                # dX = dgi W_ih: W_ih (3H x In) is the [K][N] form of the B operand
                dY = gemm_bf16_tn(dgi, wih_cat, b_mn=True)                # [M][Kl] f32
        dx = None
        if ctx.needs_input_grad[0]:
            dx = dY.view(T, Bp, -1)[:, :B, :In].transpose(0, 1).contiguous()
        ctx.saved = None
        return (dx, None, None, None, dfc_w, dfc_b) + tuple(grads)


def _gru_weights(rnn):
    ndir = 2 if rnn.bidirectional else 1
    weights = []
    for l in range(rnn.num_layers):
        for d in range(ndir):
            sfx = "_l%d%s" % (l, "_reverse" if d == 1 else "")
            if not rnn.bias:
                raise _lib.SpeechB200Error("GRU without bias is not supported")
            weights += [getattr(rnn, "weight_ih" + sfx), getattr(rnn, "weight_hh" + sfx),
                        getattr(rnn, "bias_ih" + sfx), getattr(rnn, "bias_hh" + sfx)]
    return ndir, weights


GRU_MAX_BATCH = 128   # rows one recurrence launch keeps resident (gru.cu)


def _batch_chunks(x, fn):
    """The recurrence is independent across utterances, so a minibatch larger than one launch
    holds is run as consecutive chunks of <= GRU_MAX_BATCH rows (exact, autograd sees a cat)."""
    global _announce
    if x.shape[0] <= GRU_MAX_BATCH:
        return fn(x)
    _announce = False     # several backward passes add into the same .grad: none of them is final
    try:
        return torch.cat([fn(x[i:i + GRU_MAX_BATCH])
                          for i in range(0, x.shape[0], GRU_MAX_BATCH)], 0)
    finally:
        _announce = True


def gru_stack_logits(x, rnn, fc, dropout=0.0):
    """GRU stack + sum of direction halves + output projection `fc` (an nn.Linear), fused:
    returns logits (B, T, V) - the encoder tail of CTC.forward_impl (ctc_model.py:25-32)."""
    ndir, weights = _gru_weights(rnn)
    return _batch_chunks(x, lambda xc: GRUStackFunction.apply(
        xc, ndir, rnn.hidden_size, float(dropout), fc.weight, fc.bias, *weights))


def gru_stack(x, rnn, dropout=0.0):
    """Run the sm_100a GRU stack with the parameters of an nn.GRU module (batch_first, h0 = 0)."""
    ndir, weights = _gru_weights(rnn)
    return _batch_chunks(x, lambda xc: GRUStackFunction.apply(
        xc, ndir, rnn.hidden_size, float(dropout), None, None, *weights))


class ConvStackFunction(torch.autograd.Function):
    """Conv2d+ReLU stack as im2col + tcgen05 GEMM (csrc/conv.cu, csrc/gemm.cu).

    forward(x (B,T,F) f32, specs ((kh,kw,s),...), w0, b0, w1, b1, ...) -> (B, T', C*F') f32 with
    the reference's channel-major feature order (model.py:66-71)."""

    @staticmethod
    def forward(ctx, x, specs, dropout, *params):
        """dropout > 0: nn.Dropout(p) after every ReLU (model.py:25-26) as a keep-byte mask
        (scaled by 1/(1-p)) in the activations' own layout, applied by the kernels that read them."""
        _lib.require_cuda(x, "x")
        lib = _lib.load()
        dev = x.device
        B, Ti, Fi = x.shape
        Ci = 1
        cur = x.detach().float().contiguous()
        saved = []
        masks = []
        mscale = 1.0 / (1.0 - dropout) if dropout > 0.0 else 1.0
        need_grad = any(ctx.needs_input_grad)
        sp = _lib.stream_ptr()
        for l, (kh, kw, s_) in enumerate(specs):
            w, b = params[2 * l], params[2 * l + 1]
            Co = w.shape[0]
            if Co % 8 != 0:
                raise _lib.SpeechB200Error("conv out_channels must be a multiple of 8")
            K = kh * kw * Ci
            Kp = _round_up(K, 8)
            To, Fo = (Ti - kh) // s_ + 1, (Fi - kw) // s_ + 1
            M = B * To * Fo
            A = torch.empty(M, Kp, dtype=torch.bfloat16, device=dev)
            src = cur
            mprev = masks[l - 1] if l > 0 else None
            _launch("conv_im2col", 0.0,
                    lambda: lib.sb_conv_im2col(src.data_ptr(), _lib.ptr(mprev), mscale, A.data_ptr(), B, Ti,
                                               Fi, Ci, kh, kw, s_, Kp, 1 if l > 0 else 0, sp))
            Wp = torch.zeros(Co, Kp, dtype=torch.bfloat16, device=dev)
            Wp[:, :K] = w.detach().permute(0, 2, 3, 1).reshape(Co, K)
            C = gemm_bf16_tn(A, Wp, bias=b.detach().float().contiguous())
            mask = None
            if dropout > 0.0:
                mask = (torch.rand(M, Co, device=dev) >= dropout).to(torch.uint8)
            masks.append(mask)
            if need_grad:
                saved.append((A, cur, C, Wp, (Ti, Fi, Ci, kh, kw, s_, To, Fo, Co, K, Kp)))
            cur, Ti, Fi, Ci = C, To, Fo, Co
        out = torch.empty(B, Ti, Ci * Fi, dtype=torch.float32, device=dev)
        _launch("conv_relu_to_bct", 0.0,
                lambda: lib.sb_conv_relu_to_bct(cur.data_ptr(), _lib.ptr(masks[-1]), mscale,
                                                out.data_ptr(),
                                                B, Ti, Fi, Ci, sp))
        ctx.saved = saved
        ctx.masks = masks
        ctx.mscale = mscale
        ctx.B = B
        ctx.nl = len(specs)
        return out

    @staticmethod
    def backward(ctx, dY):
        lib = _lib.load()
        dev = dY.device
        B = ctx.B
        sp = _lib.stream_ptr()
        grads = [None] * (2 * ctx.nl)
        dY = dY.contiguous().float()
        dC = None
        for l in reversed(range(ctx.nl)):
            A, Pprev, C, Wp, (Ti, Fi, Ci, kh, kw, s_, To, Fo, Co, K, Kp) = ctx.saved[l]
            M = B * To * Fo
            if dC is None:
                dC = torch.empty(M, Co, dtype=torch.bfloat16, device=dev)
                db = torch.zeros(Co, dtype=torch.float32, device=dev)
                dCl = dC
                _launch("conv_dtop", 0.0,
                        lambda: lib.sb_conv_dtop(dY.data_ptr(), C.data_ptr(),
                                                 _lib.ptr(ctx.masks[l]), ctx.mscale,
                                                 dCl.data_ptr(),
                                                 db.data_ptr(), B, To, Fo, Co, sp))
            grads[2 * l + 1] = db
            # weight gradient: contraction over the M = B*To*Fo patch rows (split-K over all SMs)
            # dWp^T [Kp][Co] = A^T dC with both operands read token-major (MN-major UMMA)
            dWpT = torch.zeros(Kp, Co, dtype=torch.float32, device=dev)
            gemm_bf16_tn(A, dC, out=dWpT, accumulate=True, a_mn=True, b_mn=True)
            dWp = dWpT.t()
            grads[2 * l] = dWp[:, :K].reshape(Co, kh, kw, Ci).permute(0, 3, 1, 2).contiguous()
            if l > 0:
                dA = gemm_bf16_tn(dC, Wp, b_mn=True)            # [M][Kp] f32 patch gradient
                Mp = B * Ti * Fi
                dCp = torch.empty(Mp, Ci, dtype=torch.bfloat16, device=dev)
                db = torch.zeros(Ci, dtype=torch.float32, device=dev)
                _launch("conv_col2im_relu", 0.0,
                        lambda: lib.sb_conv_col2im_relu(dA.data_ptr(), dA.stride(0),
                                                        Pprev.data_ptr(),
                                                        _lib.ptr(ctx.masks[l - 1]), ctx.mscale,
                                                        dCp.data_ptr(),
                                                        db.data_ptr(), B, Ti, Fi, Ci, kh, kw, s_,
                                                        sp))
                dC = dCp
        ctx.saved = None
        ctx.masks = None
        return (None, None, None) + tuple(grads)


def conv_stack(x, conv, training):
    """Conv2d+ReLU(+Dropout) front-end of the encoder (reference model.py:19-29,60-71).

    x (B, T, F) -> (B, T', C*F') with the reference's channel-major feature flattening
    (transpose(1,2) of (B,C,T',F') then view, model.py:66-71).  Runs on our im2col + tcgen05
    kernels, including the Dropout after each ReLU when training.
    """
    mods = list(conv.children())
    convs = [m for m in mods if isinstance(m, torch.nn.Conv2d)]
    ps = [m.p for m in mods if isinstance(m, torch.nn.Dropout)]
    p_drop = (ps[0] if ps else 0.0) if training else 0.0
    drop = len(set(ps)) > 1
    simple = all(c.stride[0] == c.stride[1] and c.padding == (0, 0) and c.dilation == (1, 1)
                 and c.groups == 1 and c.bias is not None and c.out_channels % 8 == 0
                 for c in convs)
    if not (convs and simple and not drop):
        raise _lib.SpeechB200Error(
            "conv_stack: unsupported convolution stack (needs square stride, no padding / "
            "dilation / groups, bias, out_channels % 8 == 0, one dropout rate); this package has "
            "no cuDNN fallback")
    specs = tuple((c.kernel_size[0], c.kernel_size[1], c.stride[0]) for c in convs)
    params = []
    for c in convs:
        params += [c.weight, c.bias]
    return ConvStackFunction.apply(x, specs, float(p_drop), *params)


def beam_topk(scores, k):
    """Top-k of a float64 CUDA score matrix in the reference's stable-sort order (score
    descending, flat index ascending).  Returns (list of flat indices, list of scores)."""
    _lib.require_cuda(scores, "scores")
    lib = _lib.load()
    sc = scores.detach().double().contiguous().reshape(-1)
    n = sc.numel()
    idx = torch.empty(k, dtype=torch.int32, device=sc.device)
    val = torch.empty(k, dtype=torch.float64, device=sc.device)
    sp = _lib.stream_ptr()
    _launch("beam_topk", 0.0,
            lambda: lib.sb_beam_topk(sc.data_ptr(), n, k, idx.data_ptr(), val.data_ptr(), sp))
    return idx.cpu().tolist(), val.cpu().tolist()


def attn_step(eh, dhx, ax_prev, conv, lin, log_t):
    """Fused NNAttention forward for the decode path (no autograd).  eh (B,T,H), dhx (B,1,H) or
    (B,H), ax_prev (B,T) or None; conv = nn.Conv1d(1,H,Kc), lin = nn.Linear(H,1).
    Returns (sx (B,1,H), ax (B,T)) like the reference module."""
    _lib.require_cuda(eh, "eh")
    lib = _lib.load()
    eh = eh.detach().float().contiguous()
    B, T, H = eh.shape
    d = dhx.detach().float().reshape(B, H).contiguous()
    axp = None if ax_prev is None else ax_prev.detach().float().contiguous()
    cw = conv.weight.detach().float().reshape(H, -1).t().contiguous()     # (Kc, H)
    Kc = cw.shape[0]
    cb = conv.bias.detach().float().contiguous()
    lw = lin.weight.detach().float().reshape(-1).contiguous()
    lb = float(lin.bias.detach().float().item()) if lin.bias is not None else 0.0
    sx = torch.empty(B, H, dtype=torch.float32, device=eh.device)
    ax = torch.empty(B, T, dtype=torch.float32, device=eh.device)
    sp = _lib.stream_ptr()
    from .functions.s2s import attn_workspace
    ws = attn_workspace(lib, B, T, H, eh.device)
    _launch("attn_step", 0.0,
            lambda: lib.sb_attn_step(eh.data_ptr(), d.data_ptr(), _lib.ptr(axp), cw.data_ptr(),
                                     cb.data_ptr(), lw.data_ptr(), lb, 1 if log_t else 0, B, T, H,
                                     Kc, sx.data_ptr(), ax.data_ptr(), ws.data_ptr(), ws.numel(),
                                     sp))
    return sx.unsqueeze(1), ax
