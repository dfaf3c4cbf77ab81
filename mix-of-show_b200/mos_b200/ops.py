"""Thin tensor-level wrappers over the C ABI (one function per kernel family).

All tensors are CUDA tensors owned by the caller; outputs are passed in (the library never allocates).
"""
import ctypes

import torch

from . import _lib
from ._lib import (MOS_ACT_NONE, MOS_ACT_RELU, MOS_OUT_BF16, MOS_OUT_F32, MOS_OUT_HEADS, GemmArgs, act_dtype, check,
                   current_stream, ptr)

BN = 160
BK = 64


def _dt(*tensors):
    return ctypes.c_int32(act_dtype(*tensors))


def gemm(A, W, out=None, *, bias=None, bias_batch=None, rows_per_batch=0, residual=None, geglu=False,
         lora_down=None, lora_up=None, lora_seg=0, conv=None, splits=1, partial=None, stages=0,
         out_f32=False, heads=None, M=None, lda=None, ldc=None, ldr=None, bias_batch_ld=0, accumulate=False,
         w_static=False, pair_mode=0, counters=None, prefetch=None, act=None):
    """out = epilogue(A @ W^T [+ LoRA]).

    A: bf16 / fp16 [M, K] (row pitch lda) or, with conv=(B, H, Wd, C), the NHWC activation [B, H, Wd, C]; the 16-bit
    outputs and the residual have A's dtype.  W: bf16 (weights) or fp16 (activations, Gram products) [N, K] (conv: [N, 9*C]).  heads: dict(seg_ptr=[...], seg_kind=[...], seg_rows_pad=[...], heads=,
    head_dim=, dpad=, dv_pad=, tokens_per_batch=) selects the head-split epilogue (Q/K rows, V transposed).
    act: None or 'relu', applied to acc + bias before the residual (16-bit row output without split-K / geglu / LoRA).
    """
    a = GemmArgs()
    a.a_dtype = act_dtype(A, residual, None if out_f32 or heads is not None else out,
                          *(heads['seg_ptr'] if heads is not None else ()))
    a.w_dtype = act_dtype(W, lora_down)
    a.A, a.W = ptr(A), ptr(W)
    N = W.shape[0]
    if conv is not None:
        B, H, Wd, C = conv
        a.conv, a.B, a.H, a.Wd, a.C = 1, B, H, Wd, C
        a.M, a.K = B * H * Wd, C
        a.lda = C if lda is None else lda
        assert W.shape[1] == 9 * C
    else:
        a.M = A.shape[0] if M is None else M
        a.K = W.shape[1]
        a.lda = (A.stride(0) if lda is None else lda)
    a.N = N
    a.splits, a.stages = splits, stages
    a.partial = ptr(partial)
    if bias is not None:
        assert bias.dtype == torch.float32
    a.bias = ptr(bias)
    a.bias_batch = ptr(bias_batch)
    a.rows_per_batch = rows_per_batch
    a.bias_batch_ld = bias_batch_ld
    a.residual = ptr(residual)
    if residual is not None:
        a.ldr = residual.stride(0) if ldr is None else ldr
    a.geglu = 1 if geglu else 0
    a.w_static = 1 if w_static else 0      # reserved (ignored by the library)
    a.pair_mode = pair_mode
    a.act = {None: MOS_ACT_NONE, 'relu': MOS_ACT_RELU}[act]
    if prefetch is not None:               # a later launch's weights: staged in L2 by this launch (no-op semantically)
        a.prefetch_ptr, a.prefetch_bytes = ptr(prefetch), prefetch.numel() * prefetch.element_size()
    if counters is not None:               # split-K with the in-kernel finalize (zeroed int32 counters, one per output tile)
        assert splits > 1 and counters.dtype == torch.int32 and out is not None
        a.tile_counters, a.tile_counters_len = ptr(counters), counters.numel()
    if lora_down is not None:
        assert lora_down.shape[0] == 16 and lora_up.dtype == torch.float32
        a.lora_down, a.lora_up = ptr(lora_down), ptr(lora_up)
        a.lora_seg = lora_seg or N
    if heads is not None:
        a.out_mode = MOS_OUT_HEADS
        for i, (p_, k_, r_) in enumerate(zip(heads['seg_ptr'], heads['seg_kind'], heads['seg_rows_pad'])):
            a.seg_ptr[i] = p_.data_ptr()
            a.seg_kind[i] = k_
            a.seg_rows_pad[i] = r_
        a.heads, a.head_dim = heads['heads'], heads['head_dim']
        a.dpad, a.dv_pad = heads['dpad'], heads['dv_pad']
        a.tokens_per_batch = heads['tokens_per_batch']
    else:
        a.out_mode = MOS_OUT_F32 if out_f32 else MOS_OUT_BF16
        a.accumulate = 1 if accumulate else 0
        a.out = ptr(out)
        if out is not None:
            a.ldc = out.stride(0) if ldc is None else ldc
    check(_lib.lib().mos_gemm_bf16(ctypes.byref(a), current_stream()), 'mos_gemm_bf16')
    return out


def pixel_unshuffle(x, y, *, r, ldy=None):
    """PixelUnshuffle(r) of fp32 NCHW x [B, C, H, W] -> 16-bit NHWC rows y [B*(H/r)*(W/r), C*r*r] (row pitch ldy)."""
    assert x.dtype == torch.float32 and x.is_contiguous()
    B, C, H, W = x.shape
    check(_lib.lib().mos_pixel_unshuffle(ptr(x), ctypes.c_int32(B), ctypes.c_int32(C), ctypes.c_int32(H), ctypes.c_int32(W),
                                         ctypes.c_int32(r), ptr(y), ctypes.c_int64(y.stride(0) if ldy is None else ldy),
                                         _dt(y), current_stream()), 'mos_pixel_unshuffle')
    return y


def avgpool2x2(x, y, *, B, H, W, C, ldx=None, ldy=None):
    """AvgPool2d(2, 2, ceil_mode=True) over 16-bit NHWC rows: x [B*H*W, ldx] -> y [B*ceil(H/2)*ceil(W/2), ldy]."""
    check(_lib.lib().mos_avgpool2x2(ptr(x), ctypes.c_int64(x.stride(0) if ldx is None else ldx), ctypes.c_int32(B),
                                    ctypes.c_int32(H), ctypes.c_int32(W), ctypes.c_int32(C), ptr(y),
                                    ctypes.c_int64(y.stride(0) if ldy is None else ldy), _dt(x, y), current_stream()),
          'mos_avgpool2x2')
    return y


def splitk_finalize(partial, splits, M, N, out, *, bias=None, bias_batch=None, rows_per_batch=0, residual=None,
                    ldc=None, ldr=None, bias_batch_ld=0):
    check(_lib.lib().mos_splitk_finalize(
        ptr(partial), ctypes.c_int32(splits), ctypes.c_int64(M), ctypes.c_int64(N), ptr(bias), ptr(bias_batch),
        ctypes.c_int64(rows_per_batch), ctypes.c_int64(bias_batch_ld), ptr(residual),
        ctypes.c_int64((residual.stride(0) if ldr is None else ldr) if residual is not None else 0), ptr(out),
        ctypes.c_int64(out.stride(0) if ldc is None else ldc), _dt(out, residual), current_stream()),
        'mos_splitk_finalize')
    return out


def _s():
    return current_stream()


def attention(Q, K, Vt, out, *, batch, heads, head_dim, nq, nk, scale=None, probs=None, ldo=None):
    """Flash attention over head-split Q/K [B*H, n, DP] and V^T [B*H, DV, nk8]; out bf16 [B, nq, ldo]."""
    scale = head_dim ** -0.5 if scale is None else scale
    check(_lib.lib().mos_attention_fwd(
        ptr(Q), ptr(K), ptr(Vt), ptr(out), ctypes.c_int64(out.stride(-2) if ldo is None else ldo), ptr(probs),
        ctypes.c_int32(batch), ctypes.c_int32(heads), ctypes.c_int32(head_dim), ctypes.c_int32(nq),
        ctypes.c_int32(nk), ctypes.c_int32(Vt.shape[-1]), ctypes.c_float(scale), _dt(Q, K, Vt, out), _s()),
        'mos_attention_fwd')
    return out


def groupnorm(x, gamma, beta, y, partial, *, B, HW, C, eps, silu, ldx=None, ldy=None):
    check(_lib.lib().mos_groupnorm_fwd(
        ptr(x), ctypes.c_int64(x.stride(-2) if ldx is None else ldx), ctypes.c_int32(B), ctypes.c_int32(HW),
        ctypes.c_int32(C), ptr(gamma), ptr(beta), ctypes.c_float(eps), ctypes.c_int32(1 if silu else 0),
        ptr(partial), ctypes.c_int32(partial.numel()), ptr(y),
        ctypes.c_int64(y.stride(-2) if ldy is None else ldy), _dt(x, y), _s()), 'mos_groupnorm_fwd')
    return y


def layernorm(x, gamma, beta, y, *, M, C, eps=1e-5, ldx=None, ldy=None):
    check(_lib.lib().mos_layernorm_fwd(
        ptr(x), ctypes.c_int64(x.stride(-2) if ldx is None else ldx), ctypes.c_int64(M), ctypes.c_int32(C),
        ptr(gamma), ptr(beta), ctypes.c_float(eps), ptr(y), ctypes.c_int64(y.stride(-2) if ldy is None else ldy),
        _dt(x, y), _s()), 'mos_layernorm_fwd')
    return y


def timestep_embedding(t, out):
    check(_lib.lib().mos_timestep_embedding(ptr(t), ctypes.c_int32(out.shape[0]), ctypes.c_int32(out.shape[1]),
                                            ptr(out), _s()), 'mos_timestep_embedding')
    return out


def gemv(x, W, bias, out, *, act_in=False, act_out=False):
    nb, K = x.shape
    check(_lib.lib().mos_gemv_bf16(ptr(x), ctypes.c_int32(nb), ctypes.c_int32(K), ptr(W), ptr(bias),
                                   ctypes.c_int32(W.shape[0]), ctypes.c_int32(int(act_in)),
                                   ctypes.c_int32(int(act_out)), ptr(out), ctypes.c_int64(out.stride(0)), _s()),
          'mos_gemv_bf16')
    return out


def conv_in(x, w, bias, y, *, ldy=None):
    B, Cin, H, W = x.shape
    check(_lib.lib().mos_conv_in(ptr(x), ctypes.c_int32(B), ctypes.c_int32(Cin), ctypes.c_int32(H), ctypes.c_int32(W),
                                 ptr(w), ptr(bias), ctypes.c_int32(w.shape[1]), ptr(y),
                                 ctypes.c_int64(w.shape[1] if ldy is None else ldy), _dt(y), _s()), 'mos_conv_in')
    return y


def conv_out(x, w, bias, y, *, B, H, W, C):
    check(_lib.lib().mos_conv_out(ptr(x), ctypes.c_int32(B), ctypes.c_int32(H), ctypes.c_int32(W), ctypes.c_int32(C),
                                  ptr(w), ptr(bias), ctypes.c_int32(w.shape[0]), ptr(y), _dt(x), _s()), 'mos_conv_out')
    return y


def upsample2x(x, y, *, B, H, W, C, ldx=None):
    check(_lib.lib().mos_upsample2x(ptr(x), ctypes.c_int64(C if ldx is None else ldx), ctypes.c_int32(B),
                                    ctypes.c_int32(H), ctypes.c_int32(W), ctypes.c_int32(C), ptr(y), _s()),
          'mos_upsample2x')
    return y


def im2col_s2(x, col, *, B, H, W, C, ldx=None, pad=1):
    check(_lib.lib().mos_im2col_s2(ptr(x), ctypes.c_int64(C if ldx is None else ldx), ctypes.c_int32(B),
                                   ctypes.c_int32(H), ctypes.c_int32(W), ctypes.c_int32(C), ctypes.c_int32(pad), ptr(col),
                                   _s()), 'mos_im2col_s2')
    return col


# ----------------------------------------------------------------------------------------------- VAE glue
def softmax_rows(S, out, *, rows, cols, scale):
    assert S.dtype == torch.float32
    check(_lib.lib().mos_softmax_rows(ptr(S), ctypes.c_int64(S.stride(0)), ctypes.c_int64(rows), ctypes.c_int32(cols),
                                      ctypes.c_float(scale), ptr(out), ctypes.c_int64(out.stride(0)), _dt(out), _s()),
          'mos_softmax_rows')
    return out


def conv1x1_nchw(x, w, bias, y):
    B, Cin = x.shape[0], x.shape[1]
    check(_lib.lib().mos_conv1x1_nchw(ptr(x), ctypes.c_int32(B), ctypes.c_int32(Cin), ctypes.c_int64(x[0, 0].numel()), ptr(w),
                                      ptr(bias), ctypes.c_int32(w.shape[0]), ptr(y), _s()), 'mos_conv1x1_nchw')
    return y


def vae_moments(h, w, bias, mean, logvar, *, B, HW, L, noise=None, scaling=1.0, latents=None):
    check(_lib.lib().mos_vae_moments(ptr(h), ctypes.c_int64(h.stride(0)), ctypes.c_int32(B), ctypes.c_int64(HW),
                                     ctypes.c_int32(L), ptr(w), ptr(bias), ptr(mean), ptr(logvar), ptr(noise),
                                     ctypes.c_float(scaling), ptr(latents), _dt(h), _s()), 'mos_vae_moments')


def add_rows(x, r, *, M, C, ldx, ldr):
    check(_lib.lib().mos_add_rows(ptr(x), ctypes.c_int64(ldx), ptr(r), ctypes.c_int64(ldr), ctypes.c_int64(M),
                                  ctypes.c_int32(C), _dt(x, r), _s()), 'mos_add_rows')
    return x


def cfg_dpmpp_step(noise_pred, latents, x0_prev, unet_in, *, cfg, guidance, coef, t_out=None, t_next=0.0):
    c_x, c_m0, c_m1, alpha_s, sigma_s = coef
    check(_lib.lib().mos_cfg_dpmpp_step(ptr(noise_pred), ptr(latents), ptr(x0_prev), ptr(unet_in),
                                        ctypes.c_int64(latents.numel()), ctypes.c_int32(int(cfg)),
                                        ctypes.c_float(guidance), ctypes.c_float(c_x), ctypes.c_float(c_m0),
                                        ctypes.c_float(c_m1), ctypes.c_float(alpha_s), ctypes.c_float(sigma_s),
                                        ptr(t_out), ctypes.c_int32(0 if t_out is None else t_out.numel()),
                                        ctypes.c_float(t_next), _s()),
          'mos_cfg_dpmpp_step')
    return latents


def region_combine(glob, region_ptrs_dev, boxes, out, *, B, FH, FW, C, ld):
    n = len(boxes)
    arr = (ctypes.c_int32 * (4 * max(n, 1)))()
    for i, bx in enumerate(boxes):
        for k in range(4):
            arr[4 * i + k] = int(bx[k])
    check(_lib.lib().mos_region_combine(ptr(glob), ptr(region_ptrs_dev), ctypes.c_int32(n), arr, ctypes.c_int32(B),
                                        ctypes.c_int32(FH), ctypes.c_int32(FW), ctypes.c_int32(C), ctypes.c_int64(ld),
                                        ptr(out), _dt(glob, out), _s()), 'mos_region_combine')
    return out


# ----------------------------------------------------------------------------------------------- gradient fusion
def transpose_bf16(x, out, *, rows, C, ldx=None, ldo=None):
    check(_lib.lib().mos_transpose_bf16(ptr(x), ctypes.c_int64(x.stride(0) if ldx is None else ldx),
                                        ctypes.c_int32(rows), ctypes.c_int32(C), ptr(out),
                                        ctypes.c_int64(out.stride(0) if ldo is None else ldo), _s()),
          'mos_transpose_bf16')
    return out


def gram_small(X, G, accumulate=False):
    n, d = X.shape
    check(_lib.lib().mos_gram_small(ptr(X), ctypes.c_int32(n), ctypes.c_int32(d), ptr(G),
                                    ctypes.c_int32(int(accumulate)), _s()), 'mos_gram_small')
    return G


def atb_small(X, Y, out, accumulate=False):
    n, dx = X.shape
    check(_lib.lib().mos_atb_small(ptr(X), ptr(Y), ctypes.c_int32(n), ctypes.c_int32(dx), ctypes.c_int32(Y.shape[1]),
                                   ptr(out), ctypes.c_int32(int(accumulate)), _s()), 'mos_atb_small')
    return out


def sgemm_nn(A, B, C, alpha=1.0, beta=0.0):
    M, K = A.shape
    N = B.shape[1]
    check(_lib.lib().mos_sgemm_nn(ptr(A), ptr(B), ptr(C), ctypes.c_int32(M), ctypes.c_int32(N), ctypes.c_int32(K),
                                  ctypes.c_float(alpha), ctypes.c_float(beta), _s()), 'mos_sgemm_nn')
    return C


def dgemm_mixed(A, B, C):
    M, K = A.shape
    assert A.dtype == torch.float32 and B.dtype == torch.float64 and C.dtype == torch.float64
    check(_lib.lib().mos_dgemm_mixed(ptr(A), ptr(B), ptr(C), ctypes.c_int32(M), ctypes.c_int32(B.shape[1]),
                                     ctypes.c_int32(K), _s()), 'mos_dgemm_mixed')
    return C


def ls_grad_loss(W, Y, Cm, s, f0, grad, loss, scratch):
    """grad = 2 s (Y - Cm); loss = s <W, Y - 2 Cm> + f0"""
    assert loss.dtype == torch.float64 and scratch.dtype == torch.float64 and Y.dtype == torch.float64
    check(_lib.lib().mos_ls_grad_loss(ptr(W), ptr(Y), ptr(Cm), ctypes.c_int64(W.numel()), ctypes.c_double(s),
                                      ctypes.c_double(f0), ptr(grad), ptr(loss), ptr(scratch), _s()),
          'mos_ls_grad_loss')


def vec_dot(a, b, out, scratch):
    check(_lib.lib().mos_vec_dot(ptr(a), ptr(b), ctypes.c_int64(a.numel()), ptr(out), ptr(scratch), _s()),
          'mos_vec_dot')


def vec_asum(a, out, scratch):
    check(_lib.lib().mos_vec_asum(ptr(a), ctypes.c_int64(a.numel()), ptr(out), ptr(scratch), _s()), 'mos_vec_asum')


def vec_absmax(a, out, scratch, scale=1.0):
    check(_lib.lib().mos_vec_absmax(ptr(a), ctypes.c_int64(a.numel()), ctypes.c_float(scale), ptr(out), ptr(scratch),
                                    _s()), 'mos_vec_absmax')


def lbfgs_direction(S, Y, rho, g, h_diag, d, work, partial, gtd):
    """d = -H g (two-loop recursion over the pairs S[i], Y[i], oldest first) and gtd[0] = <g, d>; no host synchronisation."""
    k = len(S)
    PtrArr = ctypes.c_void_p * max(k, 1)
    Sp, Yp = PtrArr(*[t.data_ptr() for t in S]), PtrArr(*[t.data_ptr() for t in Y])
    rh = (ctypes.c_double * max(k, 1))(*[float(r) for r in rho])
    assert work.dtype == torch.float64 and work.numel() >= k + 1 and partial.numel() >= 257
    check(_lib.lib().mos_lbfgs_direction(Sp, Yp, rh, ctypes.c_int32(k), ptr(g), ctypes.c_float(h_diag),
                                         ctypes.c_int64(g.numel()), ptr(d), ptr(work), ptr(partial), ptr(gtd), _s()),
          'mos_lbfgs_direction')
    return d


def lbfgs_solve_batch(problems, iters, workers=4, history=25):
    """problems: list of (G fp64 [in,in], R fp64 [out,in], s, f0, best_D fp32 [out*in] (written)); runs the native L-BFGS
    driver (mos_lbfgs_solve_batch: `workers` host threads x CUDA streams inside the library).  -> [(best_loss, n_evals)]."""
    from ._lib import LbfgsProblem
    n = len(problems)
    arr = (LbfgsProblem * n)()
    losses = (ctypes.c_double * n)()
    evals = (ctypes.c_int32 * n)()
    for i, (G, R, s, f0, best_D) in enumerate(problems):
        assert G.dtype == torch.float64 and R.dtype == torch.float64 and best_D.dtype == torch.float32
        assert G.is_contiguous() and R.is_contiguous() and best_D.is_contiguous() and best_D.numel() == R.numel()
        p = arr[i]
        p.G, p.R, p.best_D = ptr(G), ptr(R), ptr(best_D)
        p.out_f, p.in_f = R.shape[0], R.shape[1]
        p.s, p.f0, p.max_iter, p.history = float(s), float(f0), int(iters), int(history)
        p.best_loss = ctypes.cast(ctypes.byref(losses, i * 8), ctypes.POINTER(ctypes.c_double))
        p.n_evals = ctypes.cast(ctypes.byref(evals, i * 4), ctypes.POINTER(ctypes.c_int32))
    check(_lib.lib().mos_lbfgs_solve_batch(arr, ctypes.c_int32(n), ctypes.c_int32(workers)), 'mos_lbfgs_solve_batch')
    return [(losses[i], evals[i]) for i in range(n)]


def vec_axpby(y, x, alpha, beta=1.0):
    check(_lib.lib().mos_vec_axpby(ptr(y), ptr(x), ctypes.c_float(alpha), ctypes.c_float(beta),
                                   ctypes.c_int64(y.numel()), _s()), 'mos_vec_axpby')
    return y


def lora_merge(table_dev, n_layers, alpha):
    check(_lib.lib().mos_lora_merge(ptr(table_dev), ctypes.c_int32(n_layers), ctypes.c_float(alpha), _s()),
          'mos_lora_merge')


# ----------------------------------------------------------------------------------------------- training state
def flat_adamw_step(params, grads, exp_avg, exp_avg_sq, group_end, group_lr, *, step, beta1=0.9, beta2=0.999,
                    eps=1e-8, weight_decay=0.01, grad_scale=1.0, emb_rows=0, emb_dim=0, norm_mean_out=None):
    ge = (ctypes.c_int64 * 3)(*[int(x) for x in group_end])
    gl = (ctypes.c_float * 3)(*[float(x) for x in group_lr])
    check(_lib.lib().mos_flat_adamw_step(
        ptr(params), ptr(grads), ptr(exp_avg), ptr(exp_avg_sq), ctypes.c_int64(params.numel()), ge, gl,
        ctypes.c_float(beta1), ctypes.c_float(beta2), ctypes.c_float(eps), ctypes.c_float(weight_decay),
        ctypes.c_int64(step), ctypes.c_float(grad_scale), ctypes.c_int32(emb_rows), ctypes.c_int32(emb_dim),
        ptr(norm_mean_out), _s()), 'mos_flat_adamw_step')


# ------------------------------------------------------------------------------------------------ training step
def _i32(v):
    return ctypes.c_int32(int(v))


def _i64(v):
    return ctypes.c_int64(int(v))


def attention_train(Q, K, Vt, out, lse2, *, batch, heads, head_dim, nq, nk, scale=None, pcols=None, pos=None, ldo=None):
    scale = head_dim ** -0.5 if scale is None else scale
    check(_lib.lib().mos_attention_fwd_train(
        ptr(Q), ptr(K), ptr(Vt), ptr(out), _i64(out.stride(-2) if ldo is None else ldo), ptr(lse2), ptr(pcols),
        ptr(pos), _i32(batch), _i32(heads), _i32(head_dim), _i32(nq), _i32(nk), _i32(Vt.shape[-1]),
        ctypes.c_float(scale), _s()), 'mos_attention_fwd_train')
    return out


def attention_bwd(Q, K, V, dO, Qt, Kt, dOt, lse2, delta, dq, dk, dv, *, batch, heads, head_dim, nq, nk, scale=None,
                  gcols=None, pos=None, lddq=None, lddk=None, lddv=None, causal=False):
    scale = head_dim ** -0.5 if scale is None else scale
    check(_lib.lib().mos_attention_bwd(
        ptr(Q), ptr(K), ptr(V), ptr(dO), ptr(Qt), ptr(Kt), ptr(dOt), ptr(lse2), ptr(delta), ptr(gcols), ptr(pos),
        ptr(dq), _i64(dq.stride(-2) if lddq is None else lddq), ptr(dk), _i64(dk.stride(-2) if lddk is None else lddk),
        ptr(dv), _i64(dv.stride(-2) if lddv is None else lddv), _i32(batch), _i32(heads), _i32(head_dim), _i32(nq),
        _i32(nk), _i32(Qt.shape[-1]), _i32(Kt.shape[-1]), ctypes.c_float(scale), _i32(1 if causal else 0), _s()),
        'mos_attention_bwd')


def heads_transpose(src, dst):
    BH, R, DP = src.shape
    check(_lib.lib().mos_heads_transpose(ptr(src), _i32(BH), _i32(R), _i32(DP), _i32(dst.shape[1]), _i32(dst.shape[2]),
                                         ptr(dst), _s()), 'mos_heads_transpose')
    return dst


def attn_delta(dO, O, delta, *, batch, heads, head_dim, N, ldo=None, pcols=None, gcols=None):
    check(_lib.lib().mos_attn_delta(ptr(dO), _i32(dO.shape[-1]), ptr(O), _i64(O.stride(-2) if ldo is None else ldo),
                                    _i32(batch), _i32(heads), _i32(head_dim), _i32(N), ptr(pcols), ptr(gcols),
                                    ptr(delta), _s()), 'mos_attn_delta')
    return delta


def groupnorm_bwd(x, dy, gamma, beta, dx, workspace, *, B, HW, C, eps, silu, add=None, ldx=None, lddy=None, lddx=None,
                  ldadd=None):
    check(_lib.lib().mos_groupnorm_bwd(
        ptr(x), _i64(x.stride(-2) if ldx is None else ldx), ptr(dy), _i64(dy.stride(-2) if lddy is None else lddy),
        _i32(B), _i32(HW), _i32(C), ptr(gamma), ptr(beta), ctypes.c_float(eps), _i32(1 if silu else 0), ptr(workspace),
        _i32(workspace.numel()), ptr(add), _i64(0 if add is None else (add.stride(-2) if ldadd is None else ldadd)),
        ptr(dx), _i64(dx.stride(-2) if lddx is None else lddx), _s()), 'mos_groupnorm_bwd')
    return dx


def layernorm_bwd(x, dy, gamma, dx, *, M, C, eps=1e-5, add=None, ldx=None, lddy=None, lddx=None, ldadd=None):
    check(_lib.lib().mos_layernorm_bwd(
        ptr(x), _i64(x.stride(-2) if ldx is None else ldx), ptr(dy), _i64(dy.stride(-2) if lddy is None else lddy),
        _i64(M), _i32(C), ptr(gamma), ctypes.c_float(eps), ptr(add),
        _i64(0 if add is None else (add.stride(-2) if ldadd is None else ldadd)), ptr(dx),
        _i64(dx.stride(-2) if lddx is None else lddx), _s()), 'mos_layernorm_bwd')
    return dx


def geglu_fwd(z, y, *, M, H):
    check(_lib.lib().mos_geglu_fwd(ptr(z), _i64(z.stride(-2)), _i64(M), _i32(H), ptr(y), _i64(y.stride(-2)), _s()),
          'mos_geglu_fwd')
    return y


def geglu_bwd(z, dy, dz, *, M, H):
    check(_lib.lib().mos_geglu_bwd(ptr(z), _i64(z.stride(-2)), ptr(dy), _i64(dy.stride(-2)), _i64(M), _i32(H), ptr(dz),
                                   _i64(dz.stride(-2)), _s()), 'mos_geglu_bwd')
    return dz


def upsample2x_bwd(dy, dx, *, B, H, W, C, lddy=None, lddx=None):
    check(_lib.lib().mos_upsample2x_bwd(ptr(dy), _i64(C if lddy is None else lddy), _i32(B), _i32(H), _i32(W), _i32(C),
                                        ptr(dx), _i64(C if lddx is None else lddx), _s()), 'mos_upsample2x_bwd')
    return dx


def col2im_s2(dcol, dx, *, B, H, W, C, add=None, ldadd=None, lddx=None):
    check(_lib.lib().mos_col2im_s2(ptr(dcol), _i32(B), _i32(H), _i32(W), _i32(C), ptr(add),
                                   _i64(0 if add is None else (C if ldadd is None else ldadd)), ptr(dx),
                                   _i64(C if lddx is None else lddx), _s()), 'mos_col2im_s2')
    return dx


def conv_out_bwd(dy, w, dx, *, B, H, W, C):
    check(_lib.lib().mos_conv_out_bwd(ptr(dy), _i32(B), _i32(H), _i32(W), _i32(C), ptr(w), _i32(dy.shape[1]), ptr(dx),
                                      _s()), 'mos_conv_out_bwd')
    return dx


def masked_mse(pred, target, mask, ws, loss, dpred, *, grad_scale=1.0):
    B, Cc = pred.shape[0], pred.shape[1]
    HW = pred[0, 0].numel()
    check(_lib.lib().mos_masked_mse(ptr(pred), ptr(target), ptr(mask), _i32(B), _i32(Cc), _i32(HW),
                                    ctypes.c_float(grad_scale), ptr(ws), ptr(loss), ptr(dpred), _s()), 'mos_masked_mse')
    return loss


def add_noise(x0, noise, timesteps_i32, alphas_cumprod, out):
    B = x0.shape[0]
    check(_lib.lib().mos_add_noise(ptr(x0), ptr(noise), ptr(timesteps_i32), ptr(alphas_cumprod), _i32(B),
                                   _i64(x0[0].numel()), ptr(out), _s()), 'mos_add_noise')
    return out


def lora_grad(x, dy, down, up, alpha, workspace, d_down, d_up, *, M, K, N, ldx=None, lddy=None, accumulate=False):
    check(_lib.lib().mos_lora_grad(
        ptr(x), _i64(x.stride(-2) if ldx is None else ldx), ptr(dy), _i64(dy.stride(-2) if lddy is None else lddy),
        _i64(M), _i32(K), _i32(N), ptr(down), ptr(up), ctypes.c_float(alpha), ptr(workspace), _i64(workspace.numel()),
        _i32(1 if accumulate else 0), ptr(d_down), ptr(d_up), _s()), 'mos_lora_grad')


def attn_reg_group(pcols_list, mask, cm, stats, *, B, heads, res, full_identity, weight):
    arr = (ctypes.c_void_p * len(pcols_list))(*[t.data_ptr() for t in pcols_list])
    check(_lib.lib().mos_attn_reg_group(arr, _i32(len(pcols_list)), _i32(B), _i32(heads), _i32(res), ptr(mask),
                                        _i32(mask.shape[-2]), _i32(mask.shape[-1]), _i32(1 if full_identity else 0),
                                        ctypes.c_float(weight), ptr(cm), ptr(stats), _s()), 'mos_attn_reg_group')


def attn_reg_grad(cm, mask, stats_all, gcols, *, B, res, full_identity, weight, group, L, heads, grad_scale=1.0):
    check(_lib.lib().mos_attn_reg_grad(ptr(cm), ptr(mask), _i32(B), _i32(res), _i32(mask.shape[-2]),
                                       _i32(mask.shape[-1]), _i32(1 if full_identity else 0), ctypes.c_float(weight),
                                       ptr(stats_all), _i32(stats_all.shape[0]), _i32(group), _i32(L), _i32(heads),
                                       ctypes.c_float(grad_scale), ptr(gcols), _s()), 'mos_attn_reg_grad')


def attn_reg_total(mse, stats_all, out):
    check(_lib.lib().mos_attn_reg_total(ptr(mse), ptr(stats_all), _i32(stats_all.shape[0]), ptr(out), _s()),
          'mos_attn_reg_total')


def lora_pack(table_dev, n_modules, alpha):
    check(_lib.lib().mos_lora_pack(ptr(table_dev), _i32(n_modules), ctypes.c_float(alpha), _s()), 'mos_lora_pack')


# ----------------------------------------------------------------------------------------------- CLIP text encoder
def attention_causal(Q, K, Vt, out, *, batch, heads, head_dim, n, scale, ldo=None, lse2=None):
    """Causal self-attention over one key tile (n <= 128); layouts as `attention`; lse2 (optional) is saved for the
    backward pass."""
    check(_lib.lib().mos_attention_fwd_causal(
        ptr(Q), ptr(K), ptr(Vt), ptr(out), _i64(out.stride(-2) if ldo is None else ldo), _i32(batch), _i32(heads),
        _i32(head_dim), _i32(n), _i32(Vt.shape[-1]), ctypes.c_float(scale), ptr(lse2), _s()), 'mos_attention_fwd_causal')
    return out


def quick_gelu_fwd(x, y, *, M, C):
    check(_lib.lib().mos_quick_gelu_fwd(ptr(x), _i64(x.stride(0)), _i64(M), _i32(C), ptr(y), _i64(y.stride(0)), _s()),
          'mos_quick_gelu_fwd')
    return y


def quick_gelu_bwd(x, dy, dx, *, M, C):
    check(_lib.lib().mos_quick_gelu_bwd(ptr(x), _i64(x.stride(0)), ptr(dy), _i64(dy.stride(0)), _i64(M), _i32(C), ptr(dx),
                                        _i64(dx.stride(0)), _s()), 'mos_quick_gelu_bwd')
    return dx


def clip_embed_bwd(ids, dx, rows, out, *, C, accumulate=False):
    """out[r, :C] (+)= sum of dx[m, :C] over the positions m whose token id is rows[r] (fp32 [n_rows, C])."""
    assert ids.dtype == torch.int32 and rows.dtype == torch.int32 and out.dtype == torch.float32
    check(_lib.lib().mos_clip_embed_bwd(ptr(ids), ptr(dx), _i64(dx.stride(0)), _i64(ids.numel()), _i32(C), ptr(rows),
                                        _i32(rows.numel()), _i32(1 if accumulate else 0), ptr(out), _s()),
          'mos_clip_embed_bwd')
    return out


def clip_embed(ids, token_embedding, position_embedding, x, *, T, C):
    """x[m, :C] = token_embedding[ids[m]] + position_embedding[m % T] (bf16 rows of pitch x.stride(0), pad columns zeroed)."""
    assert ids.dtype == torch.int32 and token_embedding.dtype == torch.float32 and position_embedding.dtype == torch.float32
    check(_lib.lib().mos_clip_embed(ptr(ids), ptr(token_embedding), ptr(position_embedding), _i64(ids.numel()), _i32(T),
                                    _i32(C), _i32(token_embedding.shape[0]), ptr(x), _i64(x.stride(0)), _s()),
          'mos_clip_embed')
    return x


def quick_gelu(x, *, M, C):
    check(_lib.lib().mos_quick_gelu(ptr(x), _i64(x.stride(0)), _i64(M), _i32(C), _s()), 'mos_quick_gelu')
    return x
