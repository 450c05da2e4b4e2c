"""Fused ViT block glue over libxqb200 (csrc/vit_kernels.cu).

`run_blocks(vit, x)` walks `vit.blocks` + `vit.norm` exactly like the reference
(dino_enc/dinov2.py:183-190 -> vision_transformer.py:336-339) but replaces every chain
   [+ residual] -> LayerScale -> DropPath -> add -> LayerNorm -> cast-to-bf16
by ONE kernel (`xq_vit_residual_ln_fwd`), GELU by one bf16 kernel and attention by the tcgen05 / TMEM / TMA flash
kernels of csrc/attn_kernel.cu (`xq_vit_attn_fwd/bwd`, reading the packed qkv projection in place and writing d(qkv)
in the packed layout); the projection GEMMs stay on cuBLAS.  Attention dropout > 0 (no shipped config) and head
dims other than 64 use the SDPA library kernel.  The residual stream is fp32 and the GEMM operands bf16,
which is what bf16 autocast gives the reference, so the numerics are the reference's.
"""
from __future__ import annotations

import torch
import torch.nn as nn
import torch.nn.functional as F

from . import _capi as C
from ._capi import call as _call, lib as _lib, ptr as _ptr, stream_ptr as _stream

_SUPPORTED_D = (384, 768, 1024)


class _ResidualLN(torch.autograd.Function):
    """(x, branch, branch_bias, ls_gamma, rowscale, ln_w, ln_b) -> (x_out fp32, y bf16)
    x_out = x + rowscale * ls_gamma * (branch + branch_bias);  y = LayerNorm(x_out)."""

    @staticmethod
    def forward(ctx, x, branch, branch_bias, ls_gamma, rowscale, ln_w, ln_b, eps: float):
        Bn, S, D = x.shape
        M = Bn * S
        x = x.contiguous()
        if x.dtype != torch.float32:
            x = x.float()
        if branch is not None:
            branch = branch.contiguous()
            if branch.dtype != torch.bfloat16:
                branch = branch.to(torch.bfloat16)
        x_out = torch.empty_like(x)
        y = torch.empty(x.shape, dtype=torch.bfloat16, device=x.device)
        mean = torch.empty(M, dtype=torch.float32, device=x.device)
        rstd = torch.empty(M, dtype=torch.float32, device=x.device)
        L = C.lib()
        C.call("xq_vit_residual_ln_fwd", 1, L.xq_vit_residual_ln_fwd, C.ptr(x), C.ptr(branch), C.ptr(branch_bias),
               C.ptr(ls_gamma), C.ptr(rowscale), S, C.ptr(ln_w), C.ptr(ln_b), float(eps), M, D, C.ptr(x_out), C.ptr(y),
               C.ptr(mean), C.ptr(rstd), C.stream_ptr(x.device),
               nbytes=M * D * (10 + (2 if branch is not None else 0)))
        ctx.save_for_backward(x_out, mean, rstd, ln_w, branch, branch_bias, ls_gamma, rowscale)
        ctx.shape = (Bn, S, D)
        ctx.set_materialize_grads(False)
        return x_out, y

    @staticmethod
    def backward(ctx, g_xout, g_y):
        x_out, mean, rstd, ln_w, branch, branch_bias, ls_gamma, rowscale = ctx.saved_tensors
        Bn, S, D = ctx.shape
        M = Bn * S
        dev = x_out.device
        if g_xout is not None:
            g_xout = g_xout.contiguous()
            if g_xout.dtype != torch.float32:
                g_xout = g_xout.float()
        if g_y is not None:
            g_y = g_y.contiguous()
            if g_y.dtype != torch.bfloat16:
                g_y = g_y.to(torch.bfloat16)
        g_x = torch.empty_like(x_out)
        g_branch = torch.empty_like(branch) if branch is not None else None
        g_w = torch.empty_like(ln_w)
        g_b = torch.empty_like(ln_w)
        g_g = torch.empty_like(ls_gamma) if (branch is not None and ls_gamma is not None) else None
        g_bb = torch.empty_like(branch_bias) if (branch is not None and branch_bias is not None) else None
        L = C.lib()
        ws = C.workspace(L.xq_vit_ln_bwd_workspace_bytes(D), dev)
        C.call("xq_vit_residual_ln_bwd", 2, L.xq_vit_residual_ln_bwd, C.ptr(g_xout), C.ptr(g_y), C.ptr(x_out),
               C.ptr(mean), C.ptr(rstd), C.ptr(ln_w), C.ptr(branch), C.ptr(branch_bias), C.ptr(ls_gamma),
               C.ptr(rowscale), S, M, D, C.ptr(g_x), C.ptr(g_branch), C.ptr(g_w), C.ptr(g_b), C.ptr(g_g), C.ptr(g_bb),
               C.ptr(ws), ws.numel(), C.stream_ptr(dev),
               nbytes=M * D * (8 + (4 if g_xout is not None else 0) + (2 if g_y is not None else 0)
                               + (4 if branch is not None else 0)))
        return g_x, g_branch, g_bb, g_g, None, g_w, g_b, None


def residual_ln(x, branch, branch_bias, ls_gamma, rowscale, ln_w, ln_b, eps=1e-6):
    return _ResidualLN.apply(x, branch, branch_bias, ls_gamma, rowscale, ln_w, ln_b, eps)


class _GeluBias(torch.autograd.Function):
    """y = GELU(x + bias), x bf16 [..., C] (the fc1 GEMM output WITHOUT its bias), bias fp32 [C]."""

    @staticmethod
    def forward(ctx, x, bias):
        x = x.contiguous()
        Cc = x.shape[-1]
        M = x.numel() // Cc
        y = torch.empty_like(x)
        L = C.lib()
        C.call("xq_vit_gelu_fwd", 1, L.xq_vit_gelu_fwd, C.ptr(x), C.ptr(bias), C.ptr(y), M, Cc, C.stream_ptr(x.device),
               nbytes=M * Cc * 4)
        ctx.save_for_backward(x, bias)
        return y

    @staticmethod
    def backward(ctx, gy):
        x, bias = ctx.saved_tensors
        gy = gy.contiguous()
        if gy.dtype != torch.bfloat16:
            gy = gy.to(torch.bfloat16)
        Cc = x.shape[-1]
        M = x.numel() // Cc
        gx = torch.empty_like(x)
        gb = torch.empty_like(bias) if bias is not None else None
        L = C.lib()
        C.call("xq_vit_gelu_bwd", 1, L.xq_vit_gelu_bwd, C.ptr(x), C.ptr(bias), C.ptr(gy), C.ptr(gx), C.ptr(gb), M, Cc,
               C.stream_ptr(x.device), nbytes=M * Cc * 6)
        return gx, gb


def gelu_bias(x, bias=None):
    return _GeluBias.apply(x, bias)


MLP_TC_ENABLED = [True]       # the tcgen05 GEMMs with fused GELU / GELU' epilogues (csrc/gemm_kernel.cu)


def mlp_tc_ok(y, fc1, fc2) -> bool:
    """xq_vit_fc1_gelu_fwd / xq_vit_fc2_dgelu_bwd cover the shipped widths: bf16 tokens, hidden % 256 == 0, in- and
    out-features % 64 == 0 (the fc2 out-features are the K of the backward GEMM)."""
    return (MLP_TC_ENABLED[0] and y.is_cuda and y.dtype == torch.bfloat16 and fc1.bias is not None
            and fc1.weight.shape[0] % 256 == 0 and fc1.weight.shape[1] % 64 == 0 and fc1.weight.shape[0] // 256 <= 64
            and fc2.weight.shape[1] == fc1.weight.shape[0] and fc2.weight.shape[0] % 64 == 0)


class _FusedMLP(torch.autograd.Function):
    """branch = fc2(GELU(fc1(y)))  WITHOUT the fc2 bias (folded into the next residual_ln), timm Mlp as called from Block.forward
    (dino_enc/vision_transformer.py:336-339).  The fc1 GEMM carries bias + GELU in its epilogue, the fc2 input-gradient GEMM carries
    GELU' and the fc1-bias gradient; the other GEMMs are library calls.  Same bits as F.linear + gelu_bias (the epilogues apply
    the same device functions to the same rounded bf16 values)."""

    @staticmethod
    def forward(ctx, y, W1, b1, W2):
        K = W1.shape[1]
        N = W1.shape[0]
        y2 = y.reshape(-1, K)
        if not y2.is_contiguous():
            y2 = y2.contiguous()
        M = y2.shape[0]
        W1b = W1.to(torch.bfloat16)
        W2b = W2.to(torch.bfloat16)
        b1f = b1.float()
        pre = torch.empty(M, N, dtype=torch.bfloat16, device=y.device)
        act = torch.empty(M, N, dtype=torch.bfloat16, device=y.device)
        L = C.lib()
        C.call("xq_vit_fc1_gelu_fwd", 1, L.xq_vit_fc1_gelu_fwd, C.ptr(y2), C.ptr(W1b), C.ptr(b1f), C.ptr(pre), C.ptr(act), M, N, K,
               C.stream_ptr(y.device), nbytes=M * K * 2 + N * K * 2 + M * N * 4, nflops=2.0 * M * N * K)
        branch = act @ W2b.t()
        ctx.save_for_backward(y2, pre, act, W1b, W2b, b1f)
        ctx.out_shape = y.shape[:-1] + (W2.shape[0],)
        ctx.in_shape = y.shape
        return branch.view(ctx.out_shape)

    @staticmethod
    def backward(ctx, g):
        y2, pre, act, W1b, W2b, b1f = ctx.saved_tensors
        M, N = pre.shape
        Ko = W2b.shape[0]
        g2 = g.reshape(M, Ko)
        if g2.dtype != torch.bfloat16:
            g2 = g2.to(torch.bfloat16)
        if not g2.is_contiguous():
            g2 = g2.contiguous()
        dW2 = (g2.t() @ act).float() if ctx.needs_input_grad[3] else None
        W2t = W2b.t().contiguous()                      # [hidden, out]: the K-major B operand of d_act = g W2
        dpre = torch.empty_like(pre)
        db1 = torch.empty(N, dtype=torch.float32, device=pre.device)
        L = C.lib()
        C.call("xq_vit_fc2_dgelu_bwd", 1, L.xq_vit_fc2_dgelu_bwd, C.ptr(g2), C.ptr(W2t), C.ptr(pre), C.ptr(b1f), C.ptr(dpre), C.ptr(db1),
               M, N, Ko, C.stream_ptr(pre.device), nbytes=M * Ko * 2 + N * Ko * 2 + M * N * 4, nflops=2.0 * M * N * Ko)
        dW1 = (dpre.t() @ y2).float() if ctx.needs_input_grad[1] else None
        dy = (dpre @ W1b).view(ctx.in_shape) if ctx.needs_input_grad[0] else None
        return dy, dW1, (db1 if ctx.needs_input_grad[2] else None), dW2


def mlp_forward(mlp, y):
    """timm Mlp (fc1 -> GELU -> fc2, drop = 0) without the fc2 bias; fused tcgen05 path when the shapes allow, else library GEMMs +
    the stand-alone bias / GELU kernel."""
    if mlp_tc_ok(y, mlp.fc1, mlp.fc2):
        return _FusedMLP.apply(y, mlp.fc1.weight, mlp.fc1.bias, mlp.fc2.weight)
    h = gelu_bias(F.linear(y, mlp.fc1.weight), mlp.fc1.bias)
    return F.linear(h, mlp.fc2.weight)


ATTN_TC_ENABLED = [True]      # the tcgen05 attention kernels (csrc/attn_kernel.cu); tools flip it to time the library path


def attn_tc_ok(qkv, num_heads: int, dropout_p: float) -> bool:
    """xq_vit_attn_fwd/bwd cover what the shipped configs run: bf16, head_dim 64, no mask, attn_drop = 0."""
    return (ATTN_TC_ENABLED[0] and qkv.is_cuda and qkv.dtype == torch.bfloat16 and dropout_p == 0.0
            and qkv.shape[-1] == 3 * num_heads * 64)


def attn_tc_forward(qkv, num_heads: int):
    """qkv bf16 [B,N,3*H*64] (packed projection, read in place) -> (out bf16 [B,N,H*64], lse2 fp32 [B,H,N])."""
    B, N, C3 = qkv.shape
    qkv = qkv.contiguous()
    out = torch.empty(B, N, C3 // 3, dtype=torch.bfloat16, device=qkv.device)
    lse2 = torch.empty(B, num_heads, N, dtype=torch.float32, device=qkv.device)
    L = _lib()
    _call("xq_vit_attn_fwd", 1, L.xq_vit_attn_fwd, _ptr(qkv), _ptr(out), _ptr(lse2), B, N, num_heads, 64, 0.125,
          _stream(qkv.device), nbytes=qkv.numel() * 2 + out.numel() * 2 + lse2.numel() * 4,
          nflops=4.0 * B * num_heads * N * N * 64)
    return out, lse2


_ATTN_WS = {}


def attn_tc_backward(qkv, out, lse2, g, num_heads: int, want_bias_grad: bool = False):
    """d(out) bf16 [B,N,H*64] -> d(qkv) bf16 [B,N,3*H*64] written directly in the packed layout
    (+ its column sums = the qkv-bias gradient, fp32 [3*H*64], when asked for)."""
    B, N, C3 = qkv.shape
    g = g.contiguous()
    if g.dtype != torch.bfloat16:
        g = g.to(torch.bfloat16)
    dqkv = torch.empty_like(qkv)
    db = torch.empty(C3, dtype=torch.float32, device=qkv.device) if want_bias_grad else None
    L = _lib()
    nbytes = int(L.xq_vit_attn_bwd_workspace_bytes(B, N, num_heads))
    key = (qkv.device.index, torch.cuda.current_stream(qkv.device).cuda_stream)
    ws = _ATTN_WS.get(key)                      # one workspace per (device, stream): calls on a stream are ordered
    if ws is None or ws.numel() < nbytes:
        ws = torch.empty(nbytes, dtype=torch.uint8, device=qkv.device)
        _ATTN_WS[key] = ws
    _call("xq_vit_attn_bwd", 3, L.xq_vit_attn_bwd, _ptr(qkv), _ptr(out), _ptr(g), _ptr(lse2), _ptr(dqkv), _ptr(db), B, N, num_heads,
          64, 0.125, _ptr(ws), ws.numel(), _stream(qkv.device), nbytes=qkv.numel() * 4 + out.numel() * 4 + lse2.numel() * 4,
          nflops=10.0 * B * num_heads * N * N * 64)
    return (dqkv, db) if want_bias_grad else dqkv


def _sdpa_packed(qkv, num_heads, dropout_p):
    """q/k/v as strided views of the packed projection (no copies); returns the leaves and the library output."""
    B, N, C3 = qkv.shape
    hd = C3 // 3 // num_heads
    with torch.enable_grad():
        src = qkv.detach().view(B, N, 3, num_heads, hd)
        q = src[:, :, 0].transpose(1, 2).requires_grad_(True)
        k = src[:, :, 1].transpose(1, 2).requires_grad_(True)
        v = src[:, :, 2].transpose(1, 2).requires_grad_(True)
        out = F.scaled_dot_product_attention(q, k, v, dropout_p=dropout_p)
    return q, k, v, out


def _sdpa_packed_backward(inner, dims, g, want_bias_grad: bool):
    """d(qkv) [B,N,3C] (+ its column sums = d(bias)) from the SDPA library backward and ONE pack kernel."""
    q, k, v, out = inner
    B, N, C = dims
    H, hd = q.shape[1], q.shape[3]
    g = g.reshape(B, N, H, hd).transpose(1, 2)
    dq, dk, dv = torch.autograd.grad(out, (q, k, v), g)
    dqkv = torch.empty(B, N, 3 * C, dtype=dq.dtype, device=dq.device)
    flat = [t.transpose(1, 2) for t in (dq, dk, dv)]            # [B,N,H,hd]
    db = None
    if all(t.is_contiguous() for t in flat) and dq.dtype == torch.bfloat16:
        if want_bias_grad:
            db = torch.empty(3 * C, dtype=torch.float32, device=dq.device)
        L = _lib()
        ws = torch.empty(int(L.xq_vit_pack_workspace_bytes()), dtype=torch.uint8, device=dq.device)
        _call("xq_vit_pack_qkv", 1, L.xq_vit_pack_qkv, _ptr(flat[0]), _ptr(flat[1]), _ptr(flat[2]), _ptr(dqkv),
              _ptr(db) if db is not None else None, B * N, C, _ptr(ws), ws.numel(), _stream(dq.device),
              nbytes=B * N * C * 12)
    else:  # layout the library did not produce in our runs; keep correctness
        torch.stack([t.reshape(B, N, C) for t in flat], dim=2, out=dqkv.view(B, N, 3, C))
        if want_bias_grad:
            db = dqkv.float().sum((0, 1))
    return dqkv, db


class _PackedAttention(torch.autograd.Function):
    """softmax(q k^T / sqrt(d)) v on the packed projection qkv [B,N,3*H*hd] (vision_transformer.py:175-191).

    The attention itself is the SDPA library kernel; this wrapper only removes the layout glue autograd
    adds around it: q/k/v are strided views of the packed tensor (no copies in forward; the library
    allocates the output in [B,N,H,hd] order so the head merge is a view) and the three gradients are
    re-packed into d(qkv) by ONE vector kernel instead of stack + permute + contiguous."""

    @staticmethod
    def forward(ctx, qkv, num_heads: int, dropout_p: float):
        B, N, C3 = qkv.shape
        ctx.dims = (B, N, C3 // 3)
        ctx.tc = attn_tc_ok(qkv, num_heads, dropout_p)
        if ctx.tc:
            qkv = qkv.contiguous()
            out, lse2 = attn_tc_forward(qkv, num_heads)
            ctx.save_for_backward(qkv, out, lse2)
            ctx.heads = num_heads
            return out
        ctx.inner = _sdpa_packed(qkv, num_heads, dropout_p)
        return ctx.inner[3].detach().transpose(1, 2).reshape(B, N, C3 // 3)

    @staticmethod
    def backward(ctx, g):
        if ctx.tc:
            qkv, out, lse2 = ctx.saved_tensors
            return attn_tc_backward(qkv, out, lse2, g, ctx.heads), None, None
        inner, ctx.inner = ctx.inner, None
        dqkv, _ = _sdpa_packed_backward(inner, ctx.dims, g, False)
        return dqkv, None, None


def packed_attention(qkv, num_heads, dropout_p=0.0):
    return _PackedAttention.apply(qkv, num_heads, dropout_p)


class _QKVAttention(torch.autograd.Function):
    """qkv = y W^T + b ; attention(qkv)   (vision_transformer.py:175-191) as ONE autograd node, so that the bias
    gradient is the column sum the pack kernel already has in registers (no separate sum(0) pass over d(qkv)).
    y [B,N,C] bf16, W [3C,C] / b [3C] fp32 parameters; GEMMs are library calls in bf16 (autocast semantics)."""

    @staticmethod
    def forward(ctx, y, W, b, num_heads: int, dropout_p: float):
        B, N, C = y.shape
        Wb = W.to(torch.bfloat16)
        qkv = torch.addmm(b.to(torch.bfloat16), y.reshape(B * N, C), Wb.t()).view(B, N, 3 * C)
        ctx.dims = (B, N, C)
        ctx.tc = attn_tc_ok(qkv, num_heads, dropout_p)
        if ctx.tc:
            out, lse2 = attn_tc_forward(qkv, num_heads)
            ctx.save_for_backward(y, Wb, qkv, out, lse2)
            ctx.heads = num_heads
            return out
        ctx.inner = _sdpa_packed(qkv, num_heads, dropout_p)
        ctx.save_for_backward(y, Wb)
        return ctx.inner[3].detach().transpose(1, 2).reshape(B, N, C)

    @staticmethod
    def backward(ctx, g):
        B, N, C = ctx.dims
        if ctx.tc:
            y, Wb, qkv, out, lse2 = ctx.saved_tensors
            if ctx.needs_input_grad[2]:
                dqkv, db = attn_tc_backward(qkv, out, lse2, g, ctx.heads, want_bias_grad=True)
            else:
                dqkv, db = attn_tc_backward(qkv, out, lse2, g, ctx.heads), None
        else:
            inner, ctx.inner = ctx.inner, None
            y, Wb = ctx.saved_tensors
            dqkv, db = _sdpa_packed_backward(inner, ctx.dims, g, ctx.needs_input_grad[2])
        d2 = dqkv.view(B * N, 3 * C)
        dy = (d2 @ Wb).view(B, N, C) if ctx.needs_input_grad[0] else None
        dW = (d2.t() @ y.reshape(B * N, C)).float() if ctx.needs_input_grad[1] else None
        return dy, dW, db, None, None


def attention_forward(attn, y):
    """Attention.forward (vision_transformer.py:173-197) on the fused path (no qk_norm, no mask)."""
    if not isinstance(attn.q_norm, nn.Identity) or not isinstance(attn.k_norm, nn.Identity):
        return attn(y)
    p = attn.attn_drop.p if attn.training else 0.0
    if attn.qkv.bias is not None and y.dtype == torch.bfloat16:
        o = _QKVAttention.apply(y, attn.qkv.weight, attn.qkv.bias, attn.num_heads, p)
    else:
        o = packed_attention(attn.qkv(y), attn.num_heads, p)
    return F.linear(o, attn.proj.weight)      # the proj bias is folded into the next residual_ln


class _PatchEmbed(torch.autograd.Function):
    """timm PatchEmbed (Conv2d(kernel = stride = p) -> flatten(2).transpose(1,2)) as im2col-permutation + ONE GEMM.
    x fp32 [B,Cin,H,W] (no gradient), W [D,Cin,p,p] / b [D] fp32 parameters -> tokens bf16 [B, gh*gw, D]."""

    @staticmethod
    def forward(ctx, x, W, b):
        Bn, Cin, H, Wd = x.shape
        D, p = W.shape[0], W.shape[2]
        x = x.contiguous()
        M, K = Bn * (H // p) * (Wd // p), Cin * p * p
        patches = torch.empty(M, K, dtype=torch.bfloat16, device=x.device)
        L = _lib()
        _call("xq_vit_patchify", 1, L.xq_vit_patchify, _ptr(x), _ptr(patches), Bn, Cin, H, Wd, p, _stream(x.device),
              nbytes=x.numel() * 6)
        Wb = W.reshape(D, K).to(torch.bfloat16)
        if b is not None:
            y = torch.addmm(b.to(torch.bfloat16), patches, Wb.t())
        else:
            y = patches @ Wb.t()
        ctx.save_for_backward(patches)
        ctx.wshape = tuple(W.shape)
        ctx.has_bias = b is not None
        return y.view(Bn, M // Bn, D)

    @staticmethod
    def backward(ctx, g):
        (patches,) = ctx.saved_tensors
        D = ctx.wshape[0]
        g2 = g.reshape(-1, D)
        if g2.dtype != torch.bfloat16:
            g2 = g2.to(torch.bfloat16)
        dW = (g2.t() @ patches).float().view(ctx.wshape) if ctx.needs_input_grad[1] else None
        db = g2.float().sum(0) if (ctx.has_bias and ctx.needs_input_grad[2]) else None
        return None, dW, db


def patch_embed_ok(pe, x) -> bool:
    p = pe.patch_size[0]
    return (x.is_cuda and x.dtype == torch.float32 and not x.requires_grad and torch.is_autocast_enabled()
            and torch.get_autocast_dtype("cuda") == torch.bfloat16 and isinstance(pe.norm, nn.Identity)
            and pe.patch_size[0] == pe.patch_size[1] and p % 4 == 0 and x.shape[2] % p == 0 and x.shape[3] % p == 0
            and tuple(pe.proj.stride) == tuple(pe.proj.kernel_size) and tuple(pe.proj.padding) == (0, 0))


def patch_embed(pe, x):
    """PatchEmbed.forward on the fused path when it applies (bf16 autocast, fp32 CUDA image that needs no gradient,
    patch % 4 == 0, no norm); otherwise the module's own conv."""
    if patch_embed_ok(pe, x):
        return _PatchEmbed.apply(x, pe.proj.weight, pe.proj.bias)
    return pe(x)


class _Assemble(torch.autograd.Function):
    """out[b,t] = table[t] + (t0 <= t < t0+Ls ? src[b,t-t0] : 0)  -- the encoder / decoder token assembly as one pass."""

    @staticmethod
    def forward(ctx, src, table, t0: int):
        src = src.contiguous()
        if src.dtype not in (torch.bfloat16, torch.float32):
            src = src.float()
        table = table.float().contiguous()
        B, Ls, D = src.shape
        T = table.shape[-2]
        out = torch.empty(B, T, D, dtype=torch.float32, device=src.device)
        L = _lib()
        _call("xq_vit_assemble_fwd", 1, L.xq_vit_assemble_fwd, _ptr(src), int(src.dtype == torch.bfloat16), _ptr(table), B, Ls, T,
              D, int(t0), _ptr(out), _stream(src.device), nbytes=out.numel() * 4 + src.numel() * src.element_size())
        ctx.cfg = (B, Ls, T, D, int(t0), src.dtype, tuple(table.shape))
        return out

    @staticmethod
    def backward(ctx, g):
        B, Ls, T, D, t0, sdt, tshape = ctx.cfg
        g = g.contiguous()
        if g.dtype != torch.float32:
            g = g.float()
        d_src = torch.empty(B, Ls, D, dtype=sdt, device=g.device) if ctx.needs_input_grad[0] else None
        d_tab = torch.empty(tshape, dtype=torch.float32, device=g.device) if ctx.needs_input_grad[1] else None
        L = _lib()
        _call("xq_vit_assemble_bwd", 1, L.xq_vit_assemble_bwd, _ptr(g), B, Ls, T, D, t0, _ptr(d_src) if d_src is not None else None,
              int(sdt == torch.bfloat16), _ptr(d_tab) if d_tab is not None else None, _stream(g.device),
              nbytes=g.numel() * 4 + (d_src.numel() * d_src.element_size() if d_src is not None else 0))
        return d_src, d_tab, None


ASSEMBLE_ENABLED = [True]      # bench.py --impl eager switches the fused assembly off together with the other fused paths


def assemble_tokens(owner, path_fn, src, t0: int):
    """Token assembly through the fused kernel when it applies, else `path_fn(src)` (the module's own cat / add chain).

    `path_fn` maps the batch-dependent rows src [B,Ls,D] to the full fp32 sequence [B,T,D] and must be affine in `src` with
    the identity on rows [t0, t0+Ls) -- true for dinov2.py:151-170 / 318-336 whatever the configuration (prefix tokens,
    product quantisation, level embeddings).  That assumption is CHECKED once per module instance on a random probe; if it
    does not hold (a configuration not anticipated here) the module path is used from then on.  Active dropout on the
    sequence makes the assembly batch-dependent: module path."""
    ok = (ASSEMBLE_ENABLED[0] and src.is_cuda and src.dim() == 3 and src.shape[-1] % 4 == 0 and torch.is_autocast_enabled()
          and src.dtype in (torch.bfloat16, torch.float32))
    if ok and getattr(owner, "_assemble_ok", None) is None:
        with torch.no_grad():
            probe = torch.randn(2, src.shape[1], src.shape[2], device=src.device)
            full, base = path_fn(probe).float(), path_fn(torch.zeros_like(probe[:1])).float()
            want = base.expand(2, -1, -1).clone()
            ok_shape = base.dim() == 3 and t0 + src.shape[1] <= base.shape[1]
            if ok_shape:
                want[:, t0:t0 + src.shape[1]] += probe
            owner._assemble_ok = bool(ok_shape and torch.allclose(full, want, rtol=1e-5, atol=1e-6))
    if not ok or not owner._assemble_ok:
        return path_fn(src)
    table = path_fn(torch.zeros(1, src.shape[1], src.shape[2], dtype=torch.float32, device=src.device))[0]
    return _Assemble.apply(src, table, t0)


def _droppath_scale(mod, batch: int, device):
    """DropPath (timm): per-sample keep mask / keep_prob, or None when inactive."""
    p = getattr(mod, "drop_prob", 0.0)
    if p == 0.0 or not mod.training:
        return None
    keep = 1.0 - p
    t = torch.empty(batch, dtype=torch.float32, device=device).bernoulli_(keep)
    if keep > 0.0 and getattr(mod, "scale_by_keep", True):
        t.div_(keep)
    return t


def fused_path_ok(vit, x) -> bool:
    return (x.is_cuda and torch.is_autocast_enabled() and torch.get_autocast_dtype("cuda") == torch.bfloat16
            and vit.embed_dim in _SUPPORTED_D and isinstance(vit.norm_pre, nn.Identity))


def run_blocks(vit, x, attn_mask=None):
    """x: [B,S,D] token stream after pos-embed (fp32).  Returns norm(blocks(x)) as bf16 on the fused
    path, or the plain module path result otherwise (fp32 parity runs, CPU)."""
    if attn_mask is not None or not fused_path_ok(vit, x):
        x = x.to(torch.matmul(x.new_ones(8, 8), x.new_ones(8, 8)).dtype)   # dinov2.py:177-179
        x = vit.norm_pre(x)
        if attn_mask is not None:
            for blk in vit.blocks:
                x = blk(x, attn_mask)
        else:
            x = vit.blocks(x)
        return vit.norm(x)
    Bn = x.shape[0]
    dev = x.device
    x = x.float()
    branch = bias = gamma = rs = None
    for blk in vit.blocks:
        x, y = residual_ln(x, branch, bias, gamma, rs, blk.norm1.weight, blk.norm1.bias, blk.norm1.eps)
        plain_attn = isinstance(blk.attn.q_norm, nn.Identity) and isinstance(blk.attn.k_norm, nn.Identity)
        a = attention_forward(blk.attn, y)
        g1 = blk.ls1.gamma if hasattr(blk.ls1, "gamma") else None
        x, y = residual_ln(x, a, blk.attn.proj.bias if plain_attn else None, g1,
                           _droppath_scale(blk.drop_path1, Bn, dev), blk.norm2.weight, blk.norm2.bias, blk.norm2.eps)
        branch = mlp_forward(blk.mlp, y)          # fc1 bias in the GELU epilogue / kernel; fc2 bias folded into the next residual_ln
        bias = blk.mlp.fc2.bias
        gamma = blk.ls2.gamma if hasattr(blk.ls2, "gamma") else None
        rs = _droppath_scale(blk.drop_path2, Bn, dev)
    _, y = residual_ln(x, branch, bias, gamma, rs, vit.norm.weight, vit.norm.bias, vit.norm.eps)
    return y
