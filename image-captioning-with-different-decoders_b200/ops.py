"""Tensor-level wrappers over the C-ABI entry points (include/icd_b200.h).

torch is used here only for device memory, the current stream and dtype bookkeeping; every computation is a
kernel of libicd_b200.so.  All functions require CUDA tensors and raise otherwise — there is no CPU path.
"""
import ctypes
import os

import torch

from . import _lib
from ._lib import PREC_BF16, PREC_FP32, PREC_FP32X3, check, fill, lib, ptr, stream_ptr

_PREC = {"fp32": PREC_FP32, "bf16": PREC_BF16, "fp32x3": PREC_FP32X3}


def precision_id(p):
    if isinstance(p, int):
        return p
    return _PREC[p]


def _need_cuda(*ts):
    for t in ts:
        if t is not None and not t.is_cuda:
            raise _lib.IcdError("icd_b200 ops need CUDA tensors (got %s); there is no CPU fallback" % t.device)


def _f32c(t):
    if t.dtype != torch.float32:
        t = t.float()
    return t.contiguous()


def gemm(a, b, *, a_strides=None, b_strides=None, out=None, ldc=None, M=None, N=None, K=None,
         bias1=None, bias2=None, add1=None, ld1=0, add2=None, ld2=0, row_mask=None, beta=0.0,
         precision="fp32", flags=0):
    """C[M,N] = A[M,K] * B[N,K]^T + epilogue.  By default A is (M,K) row-major and B is (N,K) row-major
    (the nn.Linear layout: y = x W^T).  Explicit element strides (sam, sak)/(sbn, sbk) select the
    transposed forms used by the backward contractions."""
    _need_cuda(a, b)
    if a_strides is None:
        M_, K_ = a.shape
        a_strides = (a.stride(0), a.stride(1))
    if b_strides is None:
        N_, K2 = b.shape
        b_strides = (b.stride(0), b.stride(1))
    M = a.shape[0] if M is None else M
    N = b.shape[0] if N is None else N
    K = a.shape[1] if K is None else K
    if out is None:
        out = torch.empty(M, N, device=a.device, dtype=torch.float32)
        ldc = N
    elif ldc is None:
        ldc = out.stride(0)
    d = _lib.GemmDesc()
    ws = None
    need = int(lib().icd_gemm_ws_bytes(M, N, K, precision_id(precision)))
    if need:
        ws = torch.empty(need, device=a.device, dtype=torch.uint8)
    fill(d, ws=ws, ws_bytes=need)
    fill(d, A=a, sam=a_strides[0], sak=a_strides[1], B=b, sbn=b_strides[0], sbk=b_strides[1], C=out, ldc=ldc,
         M=M, N=N, K=K, bias1=bias1, bias2=bias2, add1=add1, ld1=ld1, add2=add2, ld2=ld2, row_mask=row_mask,
         beta=float(beta), precision=precision_id(precision), flags=int(flags))
    check(lib().icd_gemm(ctypes.byref(d), stream_ptr()), "icd_gemm")
    return out


def gemm_bf16(a16, b16, M, N, K, *, a_mn=False, b_mn=False, out=None, out16=None, bias1=None, add1=None, row_mask=None,
              split_k=True, want_fp32=True, ldc=None):
    """Tensor-core contraction on operands already stored in bf16 (no staging pass).  a16: (M,K) [a_mn=False] or (K,M)
    [a_mn=True] torch.bfloat16 (row stride = leading dimension, multiple of 8); b16 likewise with N.
    -> (C fp32 (M,N) or None, C16 bf16 or None)"""
    _need_cuda(a16, b16)
    assert a16.dtype == torch.bfloat16 and b16.dtype == torch.bfloat16
    dev = a16.device
    if out is None and want_fp32:
        out = torch.empty(M, N, device=dev, dtype=torch.float32)
    if ldc is None:
        ldc = out.stride(0) if out is not None else 0
    ws, nws = None, 0
    if split_k:
        nws = int(lib().icd_gemm_bf16_splitk_ws_floats(M, N, K))
        if os.environ.get("ICD_GEMM_FORCE_PLAN"):        # diagnostic plan override (tools/gemm_bench.py): room for any split
            nws = 32 * M * N
        if nws:
            ws = torch.empty(nws, device=dev, dtype=torch.float32)
    check(lib().icd_gemm_bf16_operands(ptr(a16), ctypes.c_int64(a16.stride(0)), int(a_mn), ptr(b16),
                                       ctypes.c_int64(b16.stride(0)), int(b_mn), ptr(out), ctypes.c_int64(ldc),
                                       ptr(out16), ctypes.c_int64(out16.stride(0) if out16 is not None else 0),
                                       M, N, K, ptr(bias1), ptr(add1),
                                       ctypes.c_int64(add1.stride(0) if add1 is not None else 0), ptr(row_mask),
                                       ptr(ws), ctypes.c_int64(nws), stream_ptr()), "icd_gemm_bf16_operands")
    return out, out16


def attention_step_fwd(enc, att_enc, att_dec, w_full, b_full, fbeta_pre=None, img_index=None):
    """-> (alpha (R,P), awe_raw (R,C), gate, gated)   [gate/gated None when fbeta_pre is None]"""
    _need_cuda(enc, att_enc, att_dec)
    n_img, P, C = enc.shape
    A = att_enc.shape[2]
    R = att_dec.shape[0]
    dev = enc.device
    alpha = torch.empty(R, P, device=dev, dtype=torch.float32)
    awe = torch.empty(R, C, device=dev, dtype=torch.float32)
    gate = gated = None
    if fbeta_pre is not None:
        gate = torch.empty(R, C, device=dev, dtype=torch.float32)
        gated = torch.empty(R, C, device=dev, dtype=torch.float32)
    check(lib().icd_attention_step_fwd(
        R, P, C, A, ptr(img_index), ptr(enc), ptr(att_enc), ptr(att_dec), ctypes.c_int64(att_dec.stride(0)),
        ptr(w_full), ptr(b_full), ptr(fbeta_pre), ctypes.c_int64(fbeta_pre.stride(0) if fbeta_pre is not None else 0),
        ptr(alpha), ctypes.c_int64(P), ptr(awe), ptr(gate), ptr(gated), stream_ptr()), "icd_attention_step_fwd")
    return alpha, awe, gate, gated


def attention_step_bwd(enc, att_enc, att_dec, w_full, alpha, gate, awe_raw, d_gated, d_alpha_ext=None, d_awe_out=None):
    """-> (d_att_dec (R,A), d_fbeta_pre (R,C), d_e (R,P)); d_awe_out: optional (R,C) output d_gated*gate"""
    _need_cuda(enc, att_enc, att_dec, d_gated)
    n_img, P, C = enc.shape
    A = att_enc.shape[2]
    R = att_dec.shape[0]
    dev = enc.device
    d_att_dec = torch.empty(R, A, device=dev, dtype=torch.float32)
    d_fb = torch.empty(R, C, device=dev, dtype=torch.float32)
    d_e = torch.empty(R, P, device=dev, dtype=torch.float32)
    check(lib().icd_attention_step_bwd(
        R, P, C, A, ptr(enc), ptr(att_enc), ptr(att_dec), ctypes.c_int64(att_dec.stride(0)), ptr(w_full),
        ptr(alpha), ctypes.c_int64(alpha.stride(0)),
        ptr(d_alpha_ext), ctypes.c_int64(d_alpha_ext.stride(0) if d_alpha_ext is not None else 0),
        ptr(gate), ptr(awe_raw), ptr(d_gated),
        ptr(d_att_dec), ctypes.c_int64(A), ptr(d_fb), ctypes.c_int64(C), ptr(d_e), ctypes.c_int64(P),
        ptr(d_awe_out), stream_ptr()), "icd_attention_step_bwd")
    return d_att_dec, d_fb, d_e


def attention_proj_bwd(att_enc, att_dec_all, w_full, d_e, bt):
    """att_dec_all (T,B,A) [row stride may exceed A], d_e (B,T,P), bt list[T]
    -> (d_att_enc, d_w_full, d_b_full, d_b_enc)   [d_b_enc = d_att_enc summed over (b, p): the enc_att bias gradient]"""
    B, P, A = att_enc.shape
    T = len(bt)
    dev = att_enc.device
    d_att_enc = torch.empty_like(att_enc)
    d_wf = torch.empty(A, device=dev, dtype=torch.float32)
    d_bf = torch.empty(1, device=dev, dtype=torch.float32)
    d_be = torch.empty(A, device=dev, dtype=torch.float32)
    ws = torch.empty(int(lib().icd_attention_proj_bwd_ws_floats(B, P, A)), device=dev, dtype=torch.float32)
    bt_arr = (ctypes.c_int32 * T)(*bt)
    check(lib().icd_attention_proj_bwd(B, T, P, A, bt_arr, ptr(att_enc), ptr(att_dec_all),
                                       ctypes.c_int64(att_dec_all.stride(1)), ptr(w_full), ptr(d_e),
                                       ptr(d_att_enc), ptr(d_wf), ptr(d_bf), ptr(d_be), ptr(ws), stream_ptr()),
          "icd_attention_proj_bwd")
    return d_att_enc, d_wf, d_bf, d_be


def attention_enc_grad(alphas, d_awe_all, d_mean=None, bt=None):
    """alphas (B,T,P), d_awe_all (T,B,C), d_mean (B,C) or None, bt list[T] or None
    -> d_enc (B,P,C) = sum_t alpha[b,t,p] * d_awe[t,b,c] + d_mean[b,c] / P"""
    _need_cuda(alphas, d_awe_all)
    B, T, P = alphas.shape
    C = d_awe_all.shape[2]
    dev = alphas.device
    d_enc = torch.empty(B, P, C, device=dev, dtype=torch.float32)
    bt_arr, ws = None, None
    if bt is not None:
        bt_arr = (ctypes.c_int32 * T)(*bt)
        ws = torch.empty(B, device=dev, dtype=torch.int32)
    check(lib().icd_attention_enc_grad(B, T, P, C, bt_arr, ptr(alphas.contiguous()), ptr(d_awe_all.contiguous()),
                                       ptr(d_mean), ptr(d_enc), ptr(ws), stream_ptr()), "icd_attention_enc_grad")
    return d_enc


def init_hidden_state(enc, h_w, h_b, c_w, c_b, precision="fp32"):
    _need_cuda(enc)
    B, P, C = enc.shape
    D = h_w.shape[0]
    dev = enc.device
    mean = torch.empty(B, C, device=dev, dtype=torch.float32)
    h = torch.empty(B, D, device=dev, dtype=torch.float32)
    c = torch.empty(B, D, device=dev, dtype=torch.float32)
    check(lib().icd_init_hidden_state(B, P, C, D, precision_id(precision), ptr(enc), ptr(h_w), ptr(h_b),
                                      ptr(c_w), ptr(c_b), ptr(mean), ptr(h), ptr(c), stream_ptr()),
          "icd_init_hidden_state")
    return h, c, mean


def dropout_mask(shape, p, seed, offset=0, device="cuda"):
    out = torch.empty(shape, device=device, dtype=torch.uint8)
    check(lib().icd_dropout_mask(ptr(out), ctypes.c_int64(out.numel()), ctypes.c_float(p),
                                 ctypes.c_uint64(seed), ctypes.c_uint64(offset), stream_ptr()), "icd_dropout_mask")
    return out


def clip_adam_step(param, grad, exp_avg, exp_avg_sq, step, lr=1e-4, betas=(0.9, 0.999), eps=1e-8,
                   grad_clip=5.0, grad_scale=1.0):
    _need_cuda(param, grad, exp_avg, exp_avg_sq)
    check(lib().icd_clip_adam_step(ptr(param), ptr(grad), ptr(exp_avg), ptr(exp_avg_sq),
                                   ctypes.c_int64(param.numel()), ctypes.c_float(grad_scale),
                                   ctypes.c_float(grad_clip), ctypes.c_float(lr), ctypes.c_float(betas[0]),
                                   ctypes.c_float(betas[1]), ctypes.c_float(eps), ctypes.c_int32(step),
                                   stream_ptr()), "icd_clip_adam_step")


def cross_entropy_fwd(logits, targets):
    """logits (R,V) fp32 contiguous, targets (R) int64 (<0 = ignored row) -> (row_loss (R), lse (R))"""
    _need_cuda(logits, targets)
    R, V = logits.shape
    row_loss = torch.empty(R, device=logits.device, dtype=torch.float32)
    lse = torch.empty(R, device=logits.device, dtype=torch.float32)
    check(lib().icd_cross_entropy_fwd(ctypes.c_int64(R), V, ptr(logits), ptr(targets), ptr(row_loss), ptr(lse),
                                      stream_ptr()), "icd_cross_entropy_fwd")
    return row_loss, lse


def cross_entropy_bwd(logits, targets, lse, inv_count, upstream=None, want_bf16=False, want_fp32=True, weights=None):
    """-> (d_logits (R,V) fp32 = (softmax - onehot) * inv_count * upstream, d_logits16 (R, up8(V)) bf16 or None);
    ``upstream`` is a 0-dim / 1-element CUDA fp32 tensor read on the device (no host sync).
    want_fp32=False (needs want_bf16): the fp32 gradient is NOT written — the returned fp32 tensor is allocated but
    hollow (its contents are undefined); only for callers that hand the bf16 copy on (see losses._FusedCE).
    ``weights``: optional (R,) CUDA fp32 per-row factors (icd_weighted_cross_entropy_bwd): row r is also times weights[r]."""
    _need_cuda(logits, targets, lse, weights)
    R, V = logits.shape
    assert want_fp32 or want_bf16
    d_logits = torch.empty_like(logits)
    d16, ld16 = None, 0
    if want_bf16:
        ld16 = (V + 7) // 8 * 8
        d16 = torch.empty(R, ld16, device=logits.device, dtype=torch.bfloat16)
    if weights is None:
        check(lib().icd_cross_entropy_bwd(ctypes.c_int64(R), V, ptr(logits), ptr(targets), ptr(lse), ptr(upstream),
                                          ctypes.c_float(inv_count), ptr(d_logits) if want_fp32 else None, ptr(d16),
                                          ctypes.c_int64(ld16),
                                          stream_ptr()), "icd_cross_entropy_bwd")
    else:
        assert weights.dtype == torch.float32 and weights.is_contiguous() and weights.numel() == R
        check(lib().icd_weighted_cross_entropy_bwd(ctypes.c_int64(R), V, ptr(logits), ptr(targets), ptr(lse), ptr(upstream),
                                                   ctypes.c_float(inv_count), ptr(weights),
                                                   ptr(d_logits) if want_fp32 else None, ptr(d16), ctypes.c_int64(ld16),
                                                   stream_ptr()), "icd_weighted_cross_entropy_bwd")
    return d_logits, d16


def cross_entropy_fwd_grad16(logits, targets, inv_count, weights=None):
    """Forward and bf16 gradient in one pass over the logits (icd_cross_entropy_fwd_grad16)
    -> (row_loss (R,), lse (R,), d_logits16 (R, up8(V)) bf16 = (softmax - onehot) * inv_count, NOT yet times the upstream gradient)
    ``weights``: optional (R,) CUDA fp32 per-row factors of the gradient (icd_weighted_cross_entropy_fwd_grad16); row_loss
    stays unweighted."""
    _need_cuda(logits, targets, weights)
    R, V = logits.shape
    ld16 = (V + 7) // 8 * 8
    row_loss = torch.empty(R, device=logits.device, dtype=torch.float32)
    lse = torch.empty(R, device=logits.device, dtype=torch.float32)
    d16 = torch.empty(R, ld16, device=logits.device, dtype=torch.bfloat16)
    if weights is None:
        check(lib().icd_cross_entropy_fwd_grad16(ctypes.c_int64(R), V, ptr(logits), ptr(targets), ctypes.c_float(inv_count),
                                                 ptr(row_loss), ptr(lse), ptr(d16), ctypes.c_int64(ld16), stream_ptr()),
              "icd_cross_entropy_fwd_grad16")
    else:
        assert weights.dtype == torch.float32 and weights.is_contiguous() and weights.numel() == R
        check(lib().icd_weighted_cross_entropy_fwd_grad16(ctypes.c_int64(R), V, ptr(logits), ptr(targets),
                                                          ctypes.c_float(inv_count), ptr(weights), ptr(row_loss), ptr(lse),
                                                          ptr(d16), ctypes.c_int64(ld16), stream_ptr()),
              "icd_weighted_cross_entropy_fwd_grad16")
    return row_loss, lse, d16


def scale_bf16_by_device_scalar(x16, scale):
    """x16 *= scale (1-element CUDA fp32 tensor read on the device); nothing is touched when it is exactly 1."""
    _need_cuda(x16, scale)
    check(lib().icd_scale_bf16_by_device_scalar(ptr(x16), ctypes.c_int64(x16.numel()), ptr(scale), stream_ptr()),
          "icd_scale_bf16_by_device_scalar")
    return x16


def alpha_regulariser_fwd(alphas, alpha_c):
    """models/attention.py:413-414 -> (reg 0-dim = mean_{b,p} (alpha_c - sum_t alphas)^2, resid (B,P) saved for the backward)"""
    _need_cuda(alphas)
    B, T, P = alphas.shape
    resid = torch.empty(B, P, device=alphas.device, dtype=torch.float32)
    partial = torch.empty((B * P + 255) // 256, device=alphas.device, dtype=torch.float32)
    reg = torch.empty(1, device=alphas.device, dtype=torch.float32)
    check(lib().icd_alpha_regulariser_fwd(B, T, P, ptr(alphas), ctypes.c_float(alpha_c), ptr(resid), ptr(partial), ptr(reg),
                                          stream_ptr()), "icd_alpha_regulariser_fwd")
    return reg.reshape(()), resid


def alpha_regulariser_bwd(resid, T, upstream=None):
    """-> d_alphas (B,T,P) = -2 resid / (B*P) * upstream (``upstream``: 1-element CUDA fp32 tensor read on the device)"""
    _need_cuda(resid)
    B, P = resid.shape
    d = torch.empty(B, T, P, device=resid.device, dtype=torch.float32)
    check(lib().icd_alpha_regulariser_bwd(B, T, P, ptr(resid), ptr(upstream), ptr(d), stream_ptr()), "icd_alpha_regulariser_bwd")
    return d


def cross_entropy_fwd_bwd(logits, targets, inv_count, want_grad=True):
    """Convenience: -> (row_loss (R), d_logits (R,V) = (softmax - onehot) * inv_count)"""
    row_loss, lse = cross_entropy_fwd(logits, targets)
    d_logits = cross_entropy_bwd(logits, targets, lse, inv_count)[0] if want_grad else None
    return row_loss, d_logits


def gemm_set_pair_mode(mode):
    """Force a tile-pairing mode for every eligible shape: 0 single-CTA tiles, 1 CTA pairs + TMA multicast of B,
    2 tcgen05.mma.cta_group::2 pairs; -1 restores the built-in policy.  Returns the previous forced mode (or -1)."""
    return int(lib().icd_gemm_set_pair_mode(int(mode)))


def launch_count():
    """Kernels launched by libicd_b200.so in this process so far."""
    return int(lib().icd_launch_count())


def prof_enable(on):
    """on: False/0 = off, True/1 = time every attention-step launch, n > 1 = every n-th launch of each direction."""
    check(lib().icd_prof_enable(int(on)), "icd_prof_enable")


def prof_collect():
    """-> dict(fwd_ms, fwd_launches, fwd_rows, bwd_ms, bwd_launches, bwd_rows) for the attention-step kernels."""
    f_ms, b_ms = ctypes.c_double(0), ctypes.c_double(0)
    f_n, f_r, b_n, b_r = (ctypes.c_int64(0) for _ in range(4))
    check(lib().icd_prof_collect(ctypes.byref(f_ms), ctypes.byref(f_n), ctypes.byref(f_r),
                                 ctypes.byref(b_ms), ctypes.byref(b_n), ctypes.byref(b_r)), "icd_prof_collect")
    return dict(fwd_ms=f_ms.value, fwd_launches=f_n.value, fwd_rows=f_r.value,
                bwd_ms=b_ms.value, bwd_launches=b_n.value, bwd_rows=b_r.value)


# ---- bf16-stored-feature variants (tensor-core tier) ---------------------------------------------------
def attention_step_fwd_bf16(enc16, att_enc16, att_dec, w_full, b_full, fbeta_pre=None, img_index=None):
    """enc16 (n_img,P,C) / att_enc16 (n_img,P,A) torch.bfloat16 -> (alpha, awe_raw, gate, gated, gated16)"""
    _need_cuda(enc16, att_enc16, att_dec)
    assert enc16.dtype == torch.bfloat16 and att_enc16.dtype == torch.bfloat16
    n_img, P, C = enc16.shape
    A = att_enc16.shape[2]
    R = att_dec.shape[0]
    dev = enc16.device
    alpha = torch.empty(R, P, device=dev, dtype=torch.float32)
    awe = torch.empty(R, C, device=dev, dtype=torch.float32)
    gate = gated = gated16 = None
    if fbeta_pre is not None:
        gate = torch.empty(R, C, device=dev, dtype=torch.float32)
        gated = torch.empty(R, C, device=dev, dtype=torch.float32)
        gated16 = torch.empty(R, C, device=dev, dtype=torch.bfloat16)
    check(lib().icd_attention_step_fwd_bf16(
        R, P, C, A, ptr(img_index), ptr(enc16), ptr(att_enc16), ptr(att_dec), ctypes.c_int64(att_dec.stride(0)),
        ptr(w_full), ptr(b_full), ptr(fbeta_pre), ctypes.c_int64(fbeta_pre.stride(0) if fbeta_pre is not None else 0),
        ptr(alpha), ctypes.c_int64(P), ptr(awe), ptr(gate), ptr(gated), ptr(gated16), stream_ptr()),
        "icd_attention_step_fwd_bf16")
    return alpha, awe, gate, gated, gated16


def attention_step_bwd_bf16(enc16, att_enc16, att_dec, w_full, alpha, gate, awe_raw, d_gated, d_alpha_ext=None):
    """-> (d_att_dec (R,A), d_fbeta_pre (R,C), d_e (R,P), dz16 (R, A+C) bf16 copy of [d_att_dec | d_fbeta_pre])"""
    n_img, P, C = enc16.shape
    A = att_enc16.shape[2]
    R = att_dec.shape[0]
    dev = enc16.device
    d_att_dec = torch.empty(R, A, device=dev, dtype=torch.float32)
    d_fb = torch.empty(R, C, device=dev, dtype=torch.float32)
    d_e = torch.empty(R, P, device=dev, dtype=torch.float32)
    dz16 = torch.empty(R, A + C, device=dev, dtype=torch.bfloat16)
    check(lib().icd_attention_step_bwd_bf16(
        R, P, C, A, ptr(enc16), ptr(att_enc16), ptr(att_dec), ctypes.c_int64(att_dec.stride(0)), ptr(w_full),
        ptr(alpha), ctypes.c_int64(alpha.stride(0)),
        ptr(d_alpha_ext), ctypes.c_int64(d_alpha_ext.stride(0) if d_alpha_ext is not None else 0),
        ptr(gate), ptr(awe_raw), ptr(d_gated),
        ptr(d_att_dec), ctypes.c_int64(A), ptr(d_fb), ctypes.c_int64(C), ptr(d_e), ctypes.c_int64(P),
        ptr(dz16), ctypes.c_int64(A + C), None, stream_ptr()), "icd_attention_step_bwd_bf16")
    return d_att_dec, d_fb, d_e, dz16


def attention_proj_bwd_bf16(att_enc16, att_dec_all, w_full, d_e, bt, d_att_dec_all=None):
    """-> (d_att_enc fp32, d_att_enc16 bf16, d_w_full, d_b_full, d_b_enc).  d_att_dec_all (T, B, A): the gradient w.r.t. att_dec from
    the per-step backward kernels — switches d_w_full to its split form (icd_attention_proj_bwd_bf16_ex)."""
    B, P, A = att_enc16.shape
    T = len(bt)
    dev = att_enc16.device
    d_att_enc = torch.empty(B, P, A, device=dev, dtype=torch.float32)
    d_att_enc16 = torch.empty(B, P, A, device=dev, dtype=torch.bfloat16)
    d_wf = torch.empty(A, device=dev, dtype=torch.float32)
    d_bf = torch.empty(1, device=dev, dtype=torch.float32)
    d_be = torch.empty(A, device=dev, dtype=torch.float32)
    ws = torch.empty(int(lib().icd_attention_proj_bwd_ws_floats(B, P, A)), device=dev, dtype=torch.float32)
    bt_arr = (ctypes.c_int32 * T)(*bt)
    check(lib().icd_attention_proj_bwd_bf16_ex(B, T, P, A, bt_arr, ptr(att_enc16), ptr(att_dec_all),
                                               ctypes.c_int64(att_dec_all.stride(1)), ptr(w_full), ptr(d_e),
                                               ptr(d_att_enc), ptr(d_att_enc16), ptr(d_wf), ptr(d_bf), ptr(d_be), ptr(ws),
                                               ptr(d_att_dec_all) if d_att_dec_all is not None else None,
                                               ctypes.c_int64(d_att_dec_all.stride(1) if d_att_dec_all is not None else 0),
                                               stream_ptr()),
          "icd_attention_proj_bwd_bf16_ex")
    return d_att_enc, d_att_enc16, d_wf, d_bf, d_be


# ---- K8: the nn.LSTM recurrence as one persistent kernel per direction (csrc/lstm_persistent.cu) -----------------
def lstm_seq_supported(B, L, H):
    return bool(lib().icd_lstm_seq_supported(int(B), int(L), int(H)))


def lstm_seq_fwd(w_hh, xg):
    """w_hh (4H,H) fp32, xg (L,B,4H) fp32 = x W_ih^T + b_ih + b_hh  ->  dict(gates_act (L,B,4H), c_all, h_all (L+1,B,H),
    hout (B,L,H), hout16 (B*L,H) bf16) from a zero initial state (models/baseline.py:106)."""
    _need_cuda(w_hh, xg)
    L, B, H4 = xg.shape
    H = H4 // 4
    dev = xg.device
    f32 = dict(device=dev, dtype=torch.float32)
    out = dict(gates_act=torch.empty(L, B, 4 * H, **f32), c_all=torch.empty(L + 1, B, H, **f32),
               h_all=torch.empty(L + 1, B, H, **f32), hout=torch.empty(B, L, H, **f32),
               hout16=torch.empty(B * L, H, device=dev, dtype=torch.bfloat16))
    h16 = torch.empty((L + 1) * B, H, device=dev, dtype=torch.bfloat16)
    bar = torch.zeros(64, device=dev, dtype=torch.int32)
    check(lib().icd_lstm_seq_fwd(B, L, H, ptr(w_hh.contiguous()), ptr(xg.contiguous()), ptr(out["gates_act"]),
                                 ptr(out["c_all"]), ptr(out["h_all"]), ptr(out["hout"]), ptr(h16), ptr(out["hout16"]),
                                 ptr(bar), stream_ptr()), "icd_lstm_seq_fwd")
    out["h16"] = h16
    return out


def lstm_seq_bwd(w_hh, d_hout, gates_act, c_all):
    """-> (dg (L,B,4H) fp32, dg16 (L*B,4H) bf16): gradient w.r.t. the pre-activation gates of every step."""
    _need_cuda(w_hh, d_hout, gates_act, c_all)
    L, B, H4 = gates_act.shape
    H = H4 // 4
    dev = gates_act.device
    dg = torch.empty(L, B, 4 * H, device=dev, dtype=torch.float32)
    dg16 = torch.empty(L * B, 4 * H, device=dev, dtype=torch.bfloat16)
    dc = torch.empty(B, H, device=dev, dtype=torch.float32)
    bar = torch.zeros(64, device=dev, dtype=torch.int32)
    check(lib().icd_lstm_seq_bwd(B, L, H, ptr(w_hh.contiguous()), ptr(d_hout.contiguous()), ptr(gates_act), ptr(c_all),
                                 ptr(dc), ptr(dg), ptr(dg16), ptr(bar), stream_ptr()), "icd_lstm_seq_bwd")
    return dg, dg16
