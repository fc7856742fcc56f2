"""Tensor-level wrappers over the C ABI (one function per kernel family).

Every function takes/returns CUDA tensors and enqueues on torch's current stream.  Used by the
learner (distrl_llm_b200/learner.py) and by the parity tests, which compare each kernel with the
oracle / a plain torch fp32 reference.
"""
from __future__ import annotations

import torch

from . import _capi
from ._capi import check, lib, ptr, stream

BF16 = torch.bfloat16


def gemm(a1, b1, a2=None, b2=None, *, bias=None, residual=None, alpha=1.0, out=None,
         out_fp32=False, force_bn=0, max_ctas=0, b_mn=False):
    """C[M,N] = alpha*(a1 @ b1.T + a2 @ b2.T) + bias + residual ; a*: [M,K*], b*: [N,K*] (bf16).
    b_mn=True: the B operands are stored [K*, N] (C = a1 @ b1 + a2 @ b2), read through MN-major descriptors."""
    M, K1 = a1.shape
    N = b1.shape[1] if b_mn else b1.shape[0]
    assert (b1.shape[0] if b_mn else b1.shape[1]) == K1 and a1.dtype == BF16 and b1.dtype == BF16
    K2 = 0
    if a2 is not None:
        K2 = a2.shape[1]
        assert a2.shape[0] == M and b2.shape == ((K2, N) if b_mn else (N, K2))
    if out is None:
        out = torch.empty(M, N, device=a1.device, dtype=torch.float32 if out_fp32 else BF16)
    check(lib().b200rl_gemm(
        ptr(a1), a1.stride(0), ptr(b1), b1.stride(0), K1,
        ptr(a2), a2.stride(0) if a2 is not None else 0, ptr(b2), b2.stride(0) if b2 is not None else 0, K2,
        ptr(out), out.stride(0), 1 if out.dtype == torch.float32 else 0,
        ptr(bias), ptr(residual), residual.stride(0) if residual is not None else 0,
        float(alpha), M, N, 2 if b_mn else 0, 1, 0, force_bn, max_ctas, stream()), "gemm")
    return out


def gemm_lora(a1, b1, bext, b2, *, scale=1.0, bias=None, residual=None, b_mn=False, force_bn=0):
    """Base + LoRA projection in one launch: U = scale * a1 @ bext.T (bf16), C = a1 @ b1.T + U @ b2.T (+bias) (+residual).
    b_mn=True: dX-form layouts (b1 [K1,N], bext [K1,K2], b2 [K2,N]).  Returns (C, U)."""
    M, K1 = a1.shape
    N = b1.shape[1] if b_mn else b1.shape[0]
    K2 = bext.shape[1] if b_mn else bext.shape[0]
    assert b2.shape == ((K2, N) if b_mn else (N, K2))
    out = torch.empty(M, N, device=a1.device, dtype=BF16)
    u = torch.empty(M, K2, device=a1.device, dtype=BF16)
    check(lib().b200rl_gemm_lora(ptr(a1), a1.stride(0), ptr(b1), b1.stride(0), K1, ptr(bext), bext.stride(0), float(scale),
                                 ptr(u), u.stride(0), ptr(b2), b2.stride(0), K2, ptr(out), out.stride(0), ptr(bias),
                                 ptr(residual), residual.stride(0) if residual is not None else 0, M, N, 2 if b_mn else 0,
                                 force_bn, stream()), "gemm_lora")
    return out, u


def gemm_nf4(a1, packed, absmax, N, a2=None, b2=None, *, bias=None, residual=None, b_mn=False, force_bn=0):
    """C = a1 @ dequant(W).T (+ a2 @ b2.T): W given as NF4 storage (nf4_quantize of W [N, K1], or of W [K1, N] with
    b_mn=True), expanded inside the GEMM mainloop."""
    M, K1 = a1.shape
    K2 = a2.shape[1] if a2 is not None else 0
    out = torch.empty(M, N, device=a1.device, dtype=BF16)
    check(lib().b200rl_gemm_nf4(ptr(a1), a1.stride(0), ptr(packed), ptr(absmax), K1, ptr(a2),
                                a2.stride(0) if a2 is not None else 0, ptr(b2), b2.stride(0) if b2 is not None else 0, K2,
                                ptr(out), out.stride(0), ptr(bias), ptr(residual),
                                residual.stride(0) if residual is not None else 0, M, N, 2 if b_mn else 0, force_bn,
                                stream()), "gemm_nf4")
    return out


def gemm_dw(y, u, *, splits=1, force_bn=0):
    """dW form: returns fp32 slabs [splits, Ny, Nu] whose sum over dim 0 is y.T @ u.
    y: [tokens, Ny], u: [tokens, Nu] (bf16, row-major)."""
    Kt, Ny = y.shape
    Nu = u.shape[1]
    assert u.shape[0] == Kt and y.dtype == BF16 and u.dtype == BF16
    kb = (Kt + 63) // 64
    splits = max(1, min(splits, kb))
    per = (kb + splits - 1) // splits
    splits = (kb + per - 1) // per
    out = torch.empty(splits, Ny, Nu, device=y.device, dtype=torch.float32)
    check(lib().b200rl_gemm(
        ptr(y), y.stride(0), ptr(u), u.stride(0), Kt, None, 0, None, 0, 0,
        ptr(out), Nu, 1, None, None, 0, 1.0, Ny, Nu, 3, splits, Ny * Nu, force_bn, 0, stream()), "gemm_dw")
    return out


def embed(ids, table):
    M = ids.numel()
    out = torch.empty(M, table.shape[1], device=table.device, dtype=BF16)
    check(lib().b200rl_embed(ptr(ids), ptr(table), ptr(out), M, table.shape[1], table.shape[0], stream()), "embed")
    return out


def rmsnorm_fwd(x, w, eps):
    M, H = x.shape
    y = torch.empty_like(x)
    rstd = torch.empty(M, device=x.device, dtype=torch.float32)
    check(lib().b200rl_rmsnorm_fwd(ptr(x), ptr(w), ptr(y), ptr(rstd), M, H, float(eps), stream()), "rmsnorm_fwd")
    return y, rstd


def rmsnorm_bwd(dy, x, w, rstd, dres=None):
    M, H = x.shape
    dx = torch.empty_like(x)
    check(lib().b200rl_rmsnorm_bwd(ptr(dy), ptr(x), ptr(w), ptr(rstd), ptr(dres), ptr(dx), M, H, stream()), "rmsnorm_bwd")
    return dx


def rope_table(L, head_dim, theta, device):
    cs = torch.empty(L, head_dim // 2, 2, device=device, dtype=torch.float32)
    check(lib().b200rl_rope_table(ptr(cs), L, head_dim, float(theta), stream()), "rope_table")
    return cs


def rope_(qkv, cs, L, n_rot_heads, head_dim, backward=False):
    M = qkv.shape[0]
    check(lib().b200rl_rope(ptr(qkv), ptr(cs), M, L, qkv.stride(0), n_rot_heads, head_dim,
                            1 if backward else 0, stream()), "rope")
    return qkv


def swiglu_fwd(gu):
    M, I2 = gu.shape
    act = torch.empty(M, I2 // 2, device=gu.device, dtype=BF16)
    check(lib().b200rl_swiglu_fwd(ptr(gu), ptr(act), M, I2 // 2, stream()), "swiglu_fwd")
    return act


def swiglu_bwd(gu, dact):
    M, I2 = gu.shape
    dgu = torch.empty_like(gu)
    check(lib().b200rl_swiglu_bwd(ptr(gu), ptr(dact), ptr(dgu), M, I2 // 2, stream()), "swiglu_bwd")
    return dgu


def attn_fwd(qkv, key_mask, B, L, nq, nkv, hd, scale=None):
    scale = scale if scale is not None else hd ** -0.5
    out = torch.empty(B * L, nq * hd, device=qkv.device, dtype=BF16)
    lse = torch.empty(B, nq, L, device=qkv.device, dtype=torch.float32)
    check(lib().b200rl_attn_fwd(ptr(qkv), ptr(key_mask), ptr(out), ptr(lse), B, L, nq, nkv, hd,
                                float(scale), stream()), "attn_fwd")
    return out, lse


def attn_bwd(qkv, key_mask, out, dout, lse, B, L, nq, nkv, hd, scale=None):
    scale = scale if scale is not None else hd ** -0.5
    dqkv = torch.empty_like(qkv)
    delta = torch.empty(B, nq, L, device=qkv.device, dtype=torch.float32)
    check(lib().b200rl_attn_bwd(ptr(qkv), ptr(key_mask), ptr(out), ptr(dout), ptr(lse), ptr(delta),
                                ptr(dqkv), B, L, nq, nkv, hd, float(scale), stream()), "attn_bwd")
    return dqkv


def logprob(logits, targets, coef=None, write_grad=False):
    """Per-row log-prob of the target token; with write_grad the logits are overwritten in place by
    coef * (onehot - softmax)."""
    rows, V = logits.shape
    lp = torch.empty(rows, device=logits.device, dtype=torch.float32)
    check(lib().b200rl_logprob(ptr(logits), logits.stride(0), ptr(targets), ptr(coef), ptr(lp), rows, V,
                               1 if write_grad else 0, stream()), "logprob")
    return lp


def logprob_entropy(logits, targets, coef=None, write_grad=False, *, klw=None, ref_lp=None, old_lp=None, clip_eps=0.0,
                    slot=None, mask=None, lens=None, T=None, Bm=0, nb=1, alpha=0.0, n_slots=None):
    """logprob() plus the per-token entropy H = -sum p ln p of every row (b200rl_logprob_entropy).  Returns (lp, ent),
    both [n_slots] (default: rows) and addressed through `slot` when given.  With write_grad and alpha != 0 the
    gradient of the bonus -e*H, e = alpha * mask / (lens * Bm * nb) (mask [Bm*T], lens [Bm]), is added to dlogits."""
    rows, V = logits.shape
    n = n_slots if n_slots is not None else rows
    lp = torch.zeros(n, device=logits.device, dtype=torch.float32)
    ent = torch.zeros(n, device=logits.device, dtype=torch.float32)
    check(lib().b200rl_logprob_entropy(ptr(logits), logits.stride(0), ptr(targets), ptr(coef), ptr(klw), ptr(ref_lp),
                                       ptr(old_lp), float(clip_eps), ptr(lp), rows, V, 1 if write_grad else 0, ptr(slot),
                                       ptr(mask), ptr(lens), int(Bm), int(T if T is not None else n), int(nb), float(alpha),
                                       ptr(ent), stream()), "logprob_entropy")
    return lp, ent


def loss_value_entropy(lp, mask, adv, ent, alpha, accum, grpo, ent_accum=None):
    """loss_value() plus the entropy term -alpha * mean_i(sum_t mask H / len_i); ent_accum f64[2] += {sum mask H, sum mask}."""
    Bm, T = mask.shape
    check(lib().b200rl_loss_value_entropy(ptr(lp), ptr(mask), ptr(adv), None, 0.0, None, 0.0, ptr(accum), Bm, T,
                                          1 if grpo else 0, ptr(ent), float(alpha), ptr(ent_accum), stream()),
          "loss_value_entropy")
    return accum


def loss_coef(mask, adv, nb):
    Bm, T = mask.shape
    coef = torch.empty(Bm, T, device=mask.device, dtype=torch.float32)
    lens = torch.empty(Bm, device=mask.device, dtype=torch.int32)
    check(lib().b200rl_loss_coef(ptr(mask), ptr(adv), ptr(coef), ptr(lens), Bm, T, nb, stream()), "loss_coef")
    return coef, lens


def loss_value(lp, mask, adv, accum, grpo):
    Bm, T = mask.shape
    check(lib().b200rl_loss_value(ptr(lp), ptr(mask), ptr(adv), ptr(accum), Bm, T, 1 if grpo else 0, stream()),
          "loss_value")
    return accum


def group_advantage_topk(rewards, k, grpo):
    """rewards [G, C, 2] f64 -> (values [G,C], baselines [G], topk_idx [G,k'], topk_val [G,k'])."""
    G, Cn, two = rewards.shape
    assert two == 2 and rewards.dtype == torch.float64
    kk = min(k, Cn)
    values = torch.empty(G, Cn, device=rewards.device, dtype=torch.float64)
    base = torch.empty(G, device=rewards.device, dtype=torch.float64)
    idx = torch.empty(G, kk, device=rewards.device, dtype=torch.int32)
    val = torch.empty(G, kk, device=rewards.device, dtype=torch.float64)
    check(lib().b200rl_group_advantage_topk(ptr(rewards), ptr(values), ptr(base), ptr(idx), ptr(val),
                                            G, Cn, kk, 1 if grpo else 0, stream()), "group_advantage_topk")
    return values, base, idx, val


def nf4_quantize(w):
    """w: bf16 tensor with numel % 64 == 0 -> (packed uint8 [numel/2], absmax f32 [numel/64])."""
    n = w.numel()
    packed = torch.empty(n // 2, device=w.device, dtype=torch.uint8)
    absmax = torch.empty(n // 64, device=w.device, dtype=torch.float32)
    check(lib().b200rl_nf4_quantize(ptr(w), ptr(packed), ptr(absmax), n, stream()), "nf4_quantize")
    return packed, absmax


def nf4_dequant(packed, absmax, rows, cols, transpose=False, out=None):
    if out is None:
        out = torch.empty((cols, rows) if transpose else (rows, cols), device=packed.device, dtype=BF16)
    check(lib().b200rl_nf4_dequant(ptr(packed), ptr(absmax), ptr(out), rows, cols, 1 if transpose else 0,
                                   stream()), "nf4_dequant")
    return out


def adamw_step(p, m, v, g, step, lr, beta1=0.9, beta2=0.999, eps=1e-8, weight_decay=0.0, zero_grad=True):
    """Single-learner fused Adam(W) on flat fp32 buffers (numel % 4 == 0)."""
    import ctypes as C
    n = p.numel()
    garr = (C.c_void_p * 1)(g.data_ptr())
    check(lib().b200rl_lora_reduce_adamw(ptr(p), ptr(m), ptr(v), C.cast(garr, C.c_void_p), None, 1, 0, n,
                                         step, lr, beta1, beta2, eps, weight_decay, 1 if zero_grad else 0,
                                         stream()), "adamw")
    return p
