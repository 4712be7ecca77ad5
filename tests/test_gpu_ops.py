"""GPU tier, op level: every C-ABI kernel entry point against the oracle / an fp64 torch restatement of the same op.
Tolerances (fp32 tier): 1e-5 norm-wise for contractions and pointwise ops unless stated."""
import os

import pytest
import torch

import helpers as H
from oracle import decoders as O

pytestmark = pytest.mark.gpu


def _ops():
    from icd_b200 import ops
    return ops


@pytest.mark.parametrize("M,N,K", [(1, 1, 1), (37, 131, 77), (128, 128, 16), (200, 9490, 512), (5, 2048, 300),
                                   (513, 259, 1030)])
def test_gemm_nt_matches_fp64(cuda, M, N, K):
    ops = _ops()
    g = torch.Generator().manual_seed(M * 7 + N * 3 + K)
    a = torch.randn(M, K, generator=g).to(cuda)
    b = torch.randn(N, K, generator=g).to(cuda)
    bias = torch.randn(N, generator=g).to(cuda)
    c = ops.gemm(a, b, bias1=bias)
    ref = a.double() @ b.double().t() + bias.double()
    H.assert_close_norm(c, ref, 1e-5, "gemm NT %dx%dx%d" % (M, N, K))


def test_gemm_transposed_operand_forms(cuda):
    """The three layouts the backward uses: dX = dY W (B n-contiguous), dW = dY^T X (both row-contiguous)."""
    ops = _ops()
    g = torch.Generator().manual_seed(3)
    M, N, K = 150, 70, 260
    dy = torch.randn(M, N, generator=g).to(cuda)
    w = torch.randn(N, K, generator=g).to(cuda)
    x = torch.randn(M, K, generator=g).to(cuda)
    # dX[M,K] = dY[M,N] W[N,K]:  A = dY (k-contig), B(n=k_in, k=n_out) = W[n_out*K + k_in] -> (sbn, sbk) = (1, K)
    dx = ops.gemm(dy, w, b_strides=(1, K), M=M, N=K, K=N)
    H.assert_close_norm(dx, dy.double() @ w.double(), 1e-5, "gemm NN")
    # dW[N,K] = dY^T X: A(m=n_out, k=row) = dY[row*N + n_out] -> (1, N); B(n=k_in, k=row) = X[row*K + k_in] -> (1, K)
    dw = ops.gemm(dy, x, a_strides=(1, N), b_strides=(1, K), M=N, N=K, K=M)
    H.assert_close_norm(dw, dy.double().t() @ x.double(), 1e-5, "gemm TN")
    # A row-contiguous with B k-contiguous
    at = torch.randn(K, M, generator=g).to(cuda)           # A(m,k) = at[k*M + m]
    c = ops.gemm(at, w, a_strides=(1, M), M=M, N=N, K=K)
    H.assert_close_norm(c, at.double().t() @ w.double().t(), 1e-5, "gemm TN' ")


def test_gemm_split_k_and_epilogue(cuda):
    ops = _ops()
    g = torch.Generator().manual_seed(5)
    M, N, K = 96, 200, 8192                      # few tiles, long K -> split-K path with atomics
    a = torch.randn(M, K, generator=g).to(cuda)
    b = torch.randn(N, K, generator=g).to(cuda)
    b1 = torch.randn(N, generator=g).to(cuda)
    b2 = torch.randn(N, generator=g).to(cuda)
    add1 = torch.randn(M, N + 8, generator=g).to(cuda)
    add2 = torch.randn(M, N, generator=g).to(cuda)
    mask = (torch.rand(M, generator=g) > 0.3).to(torch.uint8).to(cuda)
    c = ops.gemm(a, b, bias1=b1, bias2=b2, add1=add1, ld1=N + 8, add2=add2, ld2=N, row_mask=mask)
    ref = a.double() @ b.double().t() + b1.double() + b2.double() + add1[:, :N].double() + add2.double()
    ref = ref * mask.double().unsqueeze(1)
    H.assert_close_norm(c, ref, 1e-5, "gemm split-k epilogue")
    assert torch.all(c[mask == 0] == 0)
    # beta accumulate into a strided output slice, unaligned N
    Ms, Ns, Ks = 33, 45, 64
    a = torch.randn(Ms, Ks, generator=g).to(cuda)
    b = torch.randn(Ns, Ks, generator=g).to(cuda)
    big = torch.randn(Ms, 101, generator=g).to(cuda)
    want = big.double().clone()
    want[:, 7:7 + Ns] += a.double() @ b.double().t()
    ops.gemm(a, b, out=big[:, 7:], ldc=101, M=Ms, N=Ns, K=Ks, beta=1.0)
    H.assert_close_norm(big, want, 1e-5, "gemm beta/ldc")


@pytest.mark.parametrize("R,A,Cdim,use_index", [(3, 48, 2048, False), (7, 512, 2048, True), (1, 64, 256, False)])
def test_attention_step_fwd_bwd_matches_oracle_autograd(cuda, R, A, Cdim, use_index):
    ops = _ops()
    g = torch.Generator().manual_seed(R * 11 + A)
    P = 196
    n_img = 3 if use_index else R
    enc = torch.randn(n_img, P, Cdim, generator=g).clamp_min_(0)
    att_enc = torch.randn(n_img, P, A, generator=g) * 0.5
    att_dec = (torch.randn(R, A, generator=g) * 0.5).requires_grad_(True)
    wf = (torch.randn(A, generator=g) * 0.2).requires_grad_(True)
    bf = torch.randn(1, generator=g).requires_grad_(True)
    fb = torch.randn(R, Cdim, generator=g).requires_grad_(True)
    idx = torch.randint(0, n_img, (R,), generator=g) if use_index else torch.arange(R)
    # oracle (fp64): models/attention.py:56-60, 270-271 with att_enc / att_dec given
    e64, ae64 = enc.double()[idx], att_enc.double()[idx].requires_grad_(True)
    ad64, wf64, bf64, fb64 = (t.detach().double().requires_grad_(True) for t in (att_dec, wf, bf, fb))
    att = (torch.relu(ae64 + ad64.unsqueeze(1)) * wf64).sum(-1) + bf64
    alpha64 = torch.softmax(att, dim=1)
    awe64 = (e64 * alpha64.unsqueeze(2)).sum(1)
    gate64 = torch.sigmoid(fb64)
    gated64 = gate64 * awe64
    img_index = idx.to(torch.int32).to(cuda) if use_index else None
    alpha, awe, gate, gated = ops.attention_step_fwd(enc.to(cuda), att_enc.to(cuda), att_dec.detach().to(cuda),
                                                     wf.detach().to(cuda), bf.detach().to(cuda),
                                                     fb.detach().to(cuda), img_index)
    H.assert_close_norm(alpha, alpha64, 1e-5, "alpha")
    H.assert_close_norm(awe, awe64, 1e-5, "awe")
    H.assert_close_norm(gate, gate64, 1e-5, "gate")
    H.assert_close_norm(gated, gated64, 1e-5, "gated")
    assert torch.allclose(alpha.sum(1).cpu(), torch.ones(R), atol=1e-5)
    if use_index:
        return
    # backward: upstream gradients on gated and directly on alpha
    d_gated = torch.randn(R, Cdim, generator=g)
    d_alpha = torch.randn(R, P, generator=g)
    ((gated64 * d_gated.double()).sum() + (alpha64 * d_alpha.double()).sum()).backward()
    d_att_dec, d_fb, d_e = ops.attention_step_bwd(enc.to(cuda), att_enc.to(cuda), att_dec.detach().to(cuda),
                                                  wf.detach().to(cuda), alpha, gate, awe, d_gated.to(cuda),
                                                  d_alpha.to(cuda))
    H.assert_close_norm(d_att_dec, ad64.grad, 2e-5, "d_att_dec")
    H.assert_close_norm(d_fb, fb64.grad, 2e-5, "d_fbeta_pre")
    d_att_enc, d_wf, d_bf, d_be = ops.attention_proj_bwd(att_enc.to(cuda), att_dec.detach().to(cuda).view(1, R, A),
                                                   wf.detach().to(cuda), d_e.view(R, 1, P), [R])
    H.assert_close_norm(d_att_enc, ae64.grad, 2e-5, "d_att_enc")
    H.assert_close_norm(d_wf, wf64.grad, 2e-5, "d_w_full")
    H.assert_close_norm(d_bf, bf64.grad, 1e-4, "d_b_full", atol=1e-5)
    H.assert_close_norm(d_be, ae64.grad.sum(dim=(0, 1)), 2e-5, "d_b_enc (enc_att bias gradient)")


def test_init_hidden_state_matches_oracle(cuda):
    ops = _ops()
    g = torch.Generator().manual_seed(9)
    B, P, C, D = 5, 196, 2048, 64
    enc = torch.randn(B, P, C, generator=g).clamp_min_(0)
    w = {"h_lin.weight": torch.randn(D, C, generator=g) * 0.02, "h_lin.bias": torch.randn(D, generator=g),
         "c_lin.weight": torch.randn(D, C, generator=g) * 0.02, "c_lin.bias": torch.randn(D, generator=g)}
    h64, c64 = O.init_hidden_state({k: v.double() for k, v in w.items()}, enc.double())
    h, c, mean = ops.init_hidden_state(enc.to(cuda), *(w[k].to(cuda) for k in
                                                        ("h_lin.weight", "h_lin.bias", "c_lin.weight", "c_lin.bias")))
    H.assert_close_norm(mean, enc.double().mean(1), 1e-6, "mean")
    H.assert_close_norm(h, h64, 1e-5, "h0")
    H.assert_close_norm(c, c64, 1e-5, "c0")


def test_dropout_mask_statistics_and_determinism(cuda):
    ops = _ops()
    m1 = ops.dropout_mask((24, 64, 512), 0.5, seed=1234, device=cuda)
    m2 = ops.dropout_mask((24, 64, 512), 0.5, seed=1234, device=cuda)
    m3 = ops.dropout_mask((24, 64, 512), 0.5, seed=1235, device=cuda)
    assert torch.equal(m1, m2) and not torch.equal(m1, m3)
    assert set(m1.unique().tolist()) <= {0, 1}
    assert abs(m1.float().mean().item() - 0.5) < 5e-3
    keep = ops.dropout_mask((1 << 20,), 0.2, seed=7, device=cuda).float().mean().item()
    assert abs(keep - 0.8) < 5e-3


def test_clip_adam_matches_torch_adam_with_clamp(cuda):
    ops = _ops()
    g = torch.Generator().manual_seed(2)
    p0 = torch.randn(10007, generator=g)
    p_ref = torch.nn.Parameter(p0.clone().double())
    opt = torch.optim.Adam([p_ref], lr=1e-3)
    p = p0.clone().to(cuda)
    m = torch.zeros_like(p)
    v = torch.zeros_like(p)
    for step in range(1, 6):
        grad = torch.randn(10007, generator=g) * 10.0            # many entries beyond +-5
        p_ref.grad = grad.double().clamp(-5, 5)                  # train_utils.py:12
        opt.step()
        ops.clip_adam_step(p, grad.to(cuda), m, v, step, lr=1e-3, grad_clip=5.0)
    H.assert_close_norm(p, p_ref.data, 1e-6, "adam params")


@pytest.mark.parametrize("V", [9490, 9491, 9488, 9489, 5, 2])
def test_cross_entropy_matches_torch(cuda, V):
    """V = 9490: rows alternate between 16- and 8-byte alignment; odd V: every alignment (scalar head / tail paths)."""
    ops = _ops()
    g = torch.Generator().manual_seed(4)
    R = 37
    x = torch.randn(R, V, generator=g) * 3
    t = torch.randint(0, V, (R,), generator=g)
    t[5] = -1
    t[11] = -1
    x64 = x.double().requires_grad_(True)
    valid = t >= 0
    loss64 = torch.nn.functional.cross_entropy(x64[valid], t[valid], reduction="sum")
    n = int(valid.sum())
    (loss64 / n).backward()
    row_loss, dx = ops.cross_entropy_fwd_bwd(x.to(cuda), t.to(cuda), 1.0 / n)
    assert abs(row_loss.sum().item() - loss64.item()) < 1e-5 * abs(loss64.item())
    H.assert_close_norm(dx, x64.grad, 1e-5, "d_logits")
    assert torch.all(dx[5] == 0) and torch.all(dx[11] == 0)
    # split entry points: upstream gradient read on the device + bf16 copy for the tensor-core tier
    rl, lse = ops.cross_entropy_fwd(x.to(cuda), t.to(cuda))
    up = torch.tensor([0.37], device=cuda)
    d32, d16 = ops.cross_entropy_bwd(x.to(cuda), t.to(cuda), lse, 1.0 / n, upstream=up, want_bf16=True)
    H.assert_close_norm(d32, x64.grad * 0.37, 1e-5, "d_logits * upstream")
    assert d16.shape[1] % 8 == 0 and d16.shape[1] >= x.shape[1]
    H.assert_close_norm(d16[:, :x.shape[1]].float(), x64.grad * 0.37, 4e-3, "d_logits16")
    assert torch.all(d16[:, x.shape[1]:] == 0)
    # one-pass kernel (forward + bf16 gradient, each row parked in shared memory): same loss and log-sum-exp bit for bit, the same
    # bf16 gradient as the two-kernel path with upstream 1; the upstream scalar is applied afterwards (untouched when it is 1)
    rl1, lse1, g16 = ops.cross_entropy_fwd_grad16(x.to(cuda), t.to(cuda), 1.0 / n)
    assert torch.equal(rl1, rl) and torch.equal(lse1, lse)
    _, ref16 = ops.cross_entropy_bwd(x.to(cuda), t.to(cuda), lse, 1.0 / n, upstream=torch.ones(1, device=cuda), want_bf16=True)
    assert torch.equal(g16, ref16)
    keep = g16.clone()
    ops.scale_bf16_by_device_scalar(g16, torch.ones(1, device=cuda))
    assert torch.equal(g16, keep)
    ops.scale_bf16_by_device_scalar(g16, up)
    H.assert_close_norm(g16[:, :x.shape[1]].float(), x64.grad * 0.37, 8e-3, "one-pass d_logits16 * upstream")


@pytest.mark.parametrize("M,N,K", [(128, 128, 64), (128, 256, 128), (512, 4608, 512), (300, 9490, 512),
                                   (77, 200, 300), (1000, 136, 2048), (12288, 512, 9490)])
def test_gemm_bf16_tensor_core_matches_bf16_rounded_fp64(cuda, M, N, K):
    """tcgen05/TMA tier: operands rounded to bf16, fp32 accumulation => compare with the fp64 product of the
    bf16-rounded operands (tolerance 2e-5 norm-wise: only the accumulation order differs)."""
    ops = _ops()
    g = torch.Generator().manual_seed(M + N + K)
    a = torch.randn(M, K, generator=g).to(cuda)
    b = torch.randn(N, K, generator=g).to(cuda)
    bias = torch.randn(N, generator=g).to(cuda)
    add = torch.randn(M, N, generator=g).to(cuda)
    mask = (torch.rand(M, generator=g) > 0.2).to(torch.uint8).to(cuda)
    c = ops.gemm(a, b, bias1=bias, add1=add, ld1=N, row_mask=mask, precision="bf16")
    ref = a.bfloat16().double() @ b.bfloat16().double().t() + bias.double() + add.double()
    ref = ref * mask.double().unsqueeze(1)
    H.assert_close_norm(c, ref, 2e-5, "tc gemm %dx%dx%d" % (M, N, K))
    # and against the unrounded fp64 product at bf16 tolerance
    full = (a.double() @ b.double().t() + bias.double() + add.double()) * mask.double().unsqueeze(1)
    H.assert_close_norm(c, full, 1e-2, "tc gemm vs fp64")


def test_gemm_bf16_transposed_forms_and_beta(cuda):
    ops = _ops()
    g = torch.Generator().manual_seed(8)
    M, N, K = 260, 150, 700
    dy = torch.randn(K, M, generator=g).to(cuda)          # A(m,k) = dy[k*M + m]  (row-contiguous source)
    x = torch.randn(K, N, generator=g).to(cuda)           # B(n,k) = x[k*N + n]
    c0 = torch.randn(M, N, generator=g).to(cuda)
    c = c0.clone()
    ops.gemm(dy, x, a_strides=(1, M), b_strides=(1, N), out=c, ldc=N, M=M, N=N, K=K, beta=1.0, precision="bf16")
    ref = c0.double() + dy.bfloat16().double().t() @ x.bfloat16().double()
    H.assert_close_norm(c, ref, 2e-5, "tc gemm TN beta")


def _bf16_features_case(R, A, Cdim, use_index, P):
    """P = 196 keeps the test id it had before P was a parameter."""
    ids = [R, A, Cdim, use_index] + ([] if P == 196 else ["P%d" % P])
    return pytest.param(R, A, Cdim, use_index, P, id="-".join(str(x) for x in ids))


@pytest.mark.parametrize("R,A,Cdim,use_index,P", [_bf16_features_case(*c) for c in [
    (3, 48, 2048, False, 196), (6, 512, 2048, True, 196), (2, 64, 512, False, 196), (3, 48, 264, False, 196), (2, 64, 520, False, 61),
    (3, 48, 2048, False, 1), (4, 64, 512, False, 16), (5, 48, 264, False, 31)]])
def test_attention_step_bf16_features_matches_oracle_on_rounded_features(cuda, R, A, Cdim, use_index, P):
    """bf16-STORED features, fp32 arithmetic: feeding the oracle the same bf16-rounded features must agree to fp32
    accuracy (1e-5) — the only approximation of this variant is the storage rounding of enc / att_enc.
    C = 264 / 520 (C % 256 != 0): the backward's scalar d_alpha path instead of the tensor-core one; P = 1 / 16 / 31 (< 32): the
    launcher never shares a row between two CTAs, not even under ICD_ATT_BWD_SPLIT=2."""
    ops = _ops()
    g = torch.Generator().manual_seed(R * 13 + A)
    n_img = 3 if use_index else R
    enc16 = torch.randn(n_img, P, Cdim, generator=g).clamp_min_(0).bfloat16()
    att_enc16 = (torch.randn(n_img, P, A, generator=g) * 0.5).bfloat16()
    att_dec = torch.randn(R, A, generator=g) * 0.5
    wf = torch.randn(A, generator=g) * 0.2
    bf = torch.randn(1, generator=g)
    fb = torch.randn(R, Cdim, generator=g)
    idx = torch.randint(0, n_img, (R,), generator=g) if use_index else torch.arange(R)
    e64 = enc16.double()[idx]
    ae64 = att_enc16.double()[idx].requires_grad_(True)
    ad64, wf64, bf64, fb64 = (t.double().requires_grad_(True) for t in (att_dec, wf, bf, fb))
    att = (torch.relu(ae64 + ad64.unsqueeze(1)) * wf64).sum(-1) + bf64
    alpha64 = torch.softmax(att, dim=1)
    awe64 = (e64 * alpha64.unsqueeze(2)).sum(1)
    gate64 = torch.sigmoid(fb64)
    gated64 = gate64 * awe64
    img_index = idx.to(torch.int32).to(cuda) if use_index else None
    alpha, awe, gate, gated, gated16 = ops.attention_step_fwd_bf16(
        enc16.to(cuda), att_enc16.to(cuda), att_dec.to(cuda), wf.to(cuda), bf.to(cuda), fb.to(cuda), img_index)
    H.assert_close_norm(alpha, alpha64, 1e-5, "alpha")
    H.assert_close_norm(awe, awe64, 1e-5, "awe")
    H.assert_close_norm(gated, gated64, 1e-5, "gated")
    H.assert_close_norm(gated16.float(), gated64, 4e-3, "gated16")
    if use_index:
        return
    d_gated = torch.randn(R, Cdim, generator=g)
    d_alpha = torch.randn(R, P, generator=g)
    ((gated64 * d_gated.double()).sum() + (alpha64 * d_alpha.double()).sum()).backward()
    d_att_dec, d_fb, d_e, dz16 = ops.attention_step_bwd_bf16(enc16.to(cuda), att_enc16.to(cuda), att_dec.to(cuda),
                                                            wf.to(cuda), alpha, gate, awe, d_gated.to(cuda),
                                                            d_alpha.to(cuda))
    # (P = 1: alpha is 1 and d_att_dec is 0 exactly; its rounding residue is held to an absolute 1e-6)
    tiny = 1e-6 if P == 1 else 0.0
    H.assert_close_norm(d_att_dec, ad64.grad, 2e-5, "d_att_dec", atol=tiny)
    H.assert_close_norm(d_fb, fb64.grad, 2e-5, "d_fbeta_pre")
    H.assert_close_norm(dz16[:, :A].float(), ad64.grad, 4e-3, "dz16[:, :A]", atol=tiny)
    H.assert_close_norm(dz16[:, A:].float(), fb64.grad, 4e-3, "dz16[:, A:]")
    # row-balance mode of the backward kernel: rows run as two half-row CTAs (2-CTA cluster, halves meet through distributed
    # shared memory); forced here for every row, the balance rule itself splits only the tail of a launch
    os.environ["ICD_ATT_BWD_SPLIT"] = "2"
    try:
        s_att_dec, s_fb, s_e, s_dz16 = ops.attention_step_bwd_bf16(enc16.to(cuda), att_enc16.to(cuda), att_dec.to(cuda),
                                                                  wf.to(cuda), alpha, gate, awe, d_gated.to(cuda), d_alpha.to(cuda))
    finally:
        del os.environ["ICD_ATT_BWD_SPLIT"]
    assert torch.equal(s_fb, d_fb) and torch.equal(s_dz16[:, A:], dz16[:, A:])
    H.assert_close_norm(s_att_dec, ad64.grad, 2e-5, "d_att_dec (split rows)", atol=tiny)
    H.assert_close_norm(s_e, d_e, 1e-5, "d_e (split rows)")
    H.assert_close_norm(s_dz16[:, :A].float(), ad64.grad, 4e-3, "dz16[:, :A] (split rows)", atol=tiny)
    d_att_enc, d_att_enc16, d_wf, d_bf, d_be = ops.attention_proj_bwd_bf16(att_enc16.to(cuda), att_dec.to(cuda).view(1, R, A),
                                                        wf.to(cuda), d_e.view(R, 1, P), [R])
    H.assert_close_norm(d_att_enc, ae64.grad, 2e-5, "d_att_enc", atol=tiny)
    H.assert_close_norm(d_att_enc16.float(), ae64.grad, 4e-3, "d_att_enc16", atol=tiny)
    H.assert_close_norm(d_be, ae64.grad.sum(dim=(0, 1)), 2e-5, "d_b_enc", atol=tiny)
    H.assert_close_norm(d_wf, wf64.grad, 2e-5, "d_w_full", atol=tiny)
    # split form of d_w_full (masked sums in the kernel + (sum att_dec * d_att_dec) / w afterwards): same results
    s_att_enc, s_att_enc16, s_wf, s_bf, s_be = ops.attention_proj_bwd_bf16(att_enc16.to(cuda), att_dec.to(cuda).view(1, R, A),
                                                        wf.to(cuda), d_e.view(R, 1, P), [R], d_att_dec_all=d_att_dec.view(1, R, A))
    assert torch.equal(s_att_enc, d_att_enc) and torch.equal(s_att_enc16, d_att_enc16) and torch.equal(s_be, d_be)
    H.assert_close_norm(s_wf, wf64.grad, 2e-5, "d_w_full (split form)", atol=tiny)
    # ... and a w_full with a zero entry falls back to the direct form inside the kernel
    wf0 = wf.clone(); wf0[3] = 0.0
    z_ref = ops.attention_proj_bwd_bf16(att_enc16.to(cuda), att_dec.to(cuda).view(1, R, A), wf0.to(cuda), d_e.view(R, 1, P), [R])
    z_spl = ops.attention_proj_bwd_bf16(att_enc16.to(cuda), att_dec.to(cuda).view(1, R, A), wf0.to(cuda), d_e.view(R, 1, P), [R],
                                        d_att_dec_all=d_att_dec.view(1, R, A))
    assert torch.equal(z_ref[2], z_spl[2]) and torch.isfinite(z_spl[2]).all()


@pytest.mark.parametrize("R,P,A,Cdim,use_index", [(5, 196, 512, 2048, False), (7, 196, 512, 2048, True), (3, 50, 64, 264, False), (100, 196, 512, 2048, False), (9, 61, 328, 520, False),
                                                  (150, 196, 64, 512, False), (300, 37, 48, 256, False)])
def test_attention_step_fwd_bf16_rows_shared_by_2_or_4_ctas_is_bit_identical(cuda, R, P, A, Cdim, use_index):
    """Few rows per launch: a row is shared by 2 / 4 CTAs (channel split, att_step_fwd_bf16_split_kernel).  Every output
    element is formed by the same operations in the same order as in the whole-row kernel, so all five outputs must be
    bit-identical under ICD_ATT_FWD_SPLIT = 1 / 2 / 4 and under the row-count rule (R = 5: four CTAs per row,
    R = 150: two, R = 300: one); pixel counts with and without an unrolled remainder, C / 4 not a multiple of the block."""
    ops = _ops()
    g = torch.Generator().manual_seed(R * 7 + P)
    n_img = 4 if use_index else R
    enc16 = torch.randn(n_img, P, Cdim, generator=g).clamp_min_(0).bfloat16().to(cuda)
    att_enc16 = (torch.randn(n_img, P, A, generator=g) * 0.5).bfloat16().to(cuda)
    att_dec = (torch.randn(R, A, generator=g) * 0.5).to(cuda)
    wf = (torch.randn(A, generator=g) * 0.2).to(cuda)
    bf = torch.randn(1, generator=g).to(cuda)
    fb = torch.randn(R, Cdim, generator=g).to(cuda)
    idx = torch.randint(0, n_img, (R,), generator=g).to(torch.int32).to(cuda) if use_index else None
    outs = {}
    for mode in ("1", "2", "4", None):
        if mode is None:
            os.environ.pop("ICD_ATT_FWD_SPLIT", None)
        else:
            os.environ["ICD_ATT_FWD_SPLIT"] = mode
        try:
            outs[mode] = ops.attention_step_fwd_bf16(enc16, att_enc16, att_dec, wf, bf, fb, idx)
        finally:
            os.environ.pop("ICD_ATT_FWD_SPLIT", None)
    for mode in ("2", "4", None):
        for name, a, b in zip(("alpha", "awe", "gate", "gated", "gated16"), outs["1"], outs[mode]):
            assert torch.equal(a, b), "%s differs between the whole-row kernel and ICD_ATT_FWD_SPLIT=%s" % (name, mode)
    # ... and without the gate inputs (SoftAttention.forward on its own): alpha + awe only
    os.environ["ICD_ATT_FWD_SPLIT"] = "4"
    try:
        a4 = ops.attention_step_fwd_bf16(enc16, att_enc16, att_dec, wf, bf, None, idx)
    finally:
        os.environ.pop("ICD_ATT_FWD_SPLIT", None)
    assert torch.equal(a4[0], outs["1"][0]) and torch.equal(a4[1], outs["1"][1])


@pytest.mark.parametrize("R", [20, 150, 300, 320, 470, 512])
def test_attention_step_bwd_bf16_row_sharing_rules_match_whole_rows(cuda, R):
    """The backward launcher's rules — every row as two half-row CTAs at few rows (R = 20, 150), the minimal balance form (R = 300,
    320, 470: only the rows beyond an equal number per SM), the full balance form (R = 512) — against the plain one-CTA-per-row
    launch (ICD_ATT_BWD_SPLIT=0): the channel-wise outputs are bit-identical, the pixel-split sums agree to fp32 rounding."""
    ops = _ops()
    g = torch.Generator().manual_seed(R)
    P, A, Cdim = 196, 64, 256
    enc16 = torch.randn(R, P, Cdim, generator=g).clamp_min_(0).bfloat16().to(cuda)
    att_enc16 = (torch.randn(R, P, A, generator=g) * 0.5).bfloat16().to(cuda)
    att_dec = (torch.randn(R, A, generator=g) * 0.5).to(cuda)
    wf = (torch.randn(A, generator=g) * 0.2).to(cuda)
    bf = torch.randn(1, generator=g).to(cuda)
    fb = torch.randn(R, Cdim, generator=g).to(cuda)
    d_gated = torch.randn(R, Cdim, generator=g).to(cuda)
    d_alpha = torch.randn(R, P, generator=g).to(cuda)
    alpha, awe, gate, gated, gated16 = ops.attention_step_fwd_bf16(enc16, att_enc16, att_dec, wf, bf, fb)
    os.environ["ICD_ATT_BWD_SPLIT"] = "0"
    try:
        w_att_dec, w_fb, w_e, w_dz16 = ops.attention_step_bwd_bf16(enc16, att_enc16, att_dec, wf, alpha, gate, awe, d_gated, d_alpha)
    finally:
        del os.environ["ICD_ATT_BWD_SPLIT"]
    s_att_dec, s_fb, s_e, s_dz16 = ops.attention_step_bwd_bf16(enc16, att_enc16, att_dec, wf, alpha, gate, awe, d_gated, d_alpha)
    assert torch.equal(s_fb, w_fb) and torch.equal(s_dz16[:, A:], w_dz16[:, A:])
    H.assert_close_norm(s_att_dec, w_att_dec, 2e-5, "d_att_dec")
    H.assert_close_norm(s_e, w_e, 1e-5, "d_e")
    H.assert_close_norm(s_dz16[:, :A].float(), w_att_dec, 4e-3, "dz16[:, :A]")
    if R in (20, 150, 300, 512):         # (the rules must actually have taken the shared form: some row differs in the last bits)
        assert not (torch.equal(s_att_dec, w_att_dec) and torch.equal(s_e, w_e))


@pytest.mark.parametrize("R,P,A,Cdim", [(40, 196, 512, 2048), (20, 196, 64, 256), (7, 61, 328, 512), (148, 50, 64, 256)])
def test_attention_step_bwd_bf16_128_register_instantiation_is_bit_identical(cuda, R, P, A, Cdim):
    """Launches of at most two CTAs per SM (<= 148 rows, every row as two half-row CTAs) use the 128-register instantiation of the
    backward kernel (twice the loads in flight in both streaming phases, batched pixel remainder): same operations in the same
    order, so all outputs must equal the 64-register instantiation's (ICD_ATT_BWD_DEEP=0) bit for bit."""
    ops = _ops()
    g = torch.Generator().manual_seed(R + P)
    enc16 = torch.randn(R, P, Cdim, generator=g).clamp_min_(0).bfloat16().to(cuda)
    att_enc16 = (torch.randn(R, P, A, generator=g) * 0.5).bfloat16().to(cuda)
    att_dec = (torch.randn(R, A, generator=g) * 0.5).to(cuda)
    wf = (torch.randn(A, generator=g) * 0.2).to(cuda)
    bf = torch.randn(1, generator=g).to(cuda)
    fb = torch.randn(R, Cdim, generator=g).to(cuda)
    d_gated = torch.randn(R, Cdim, generator=g).to(cuda)
    d_alpha = torch.randn(R, P, generator=g).to(cuda)
    alpha, awe, gate, gated, gated16 = ops.attention_step_fwd_bf16(enc16, att_enc16, att_dec, wf, bf, fb)
    deep = ops.attention_step_bwd_bf16(enc16, att_enc16, att_dec, wf, alpha, gate, awe, d_gated, d_alpha)
    os.environ["ICD_ATT_BWD_DEEP"] = "0"
    try:
        shallow = ops.attention_step_bwd_bf16(enc16, att_enc16, att_dec, wf, alpha, gate, awe, d_gated, d_alpha)
    finally:
        del os.environ["ICD_ATT_BWD_DEEP"]
    for name, a, b in zip(("d_att_dec", "d_fbeta_pre", "d_e", "dz16"), deep, shallow):
        assert torch.equal(a, b), name
    assert torch.isfinite(deep[0]).all() and torch.isfinite(deep[2]).all()


@pytest.fixture(params=[2, 1, 0], ids=["cta_group2_pairs", "multicast_pairs", "single_cta"])
def pair_mode(request):
    """Run under every tile-pairing mode of the tensor-core contraction (icd_gemm_set_pair_mode)."""
    ops = _ops()
    old = ops.gemm_set_pair_mode(request.param)
    yield request.param
    ops.gemm_set_pair_mode(old)


@pytest.mark.parametrize("N", [9490, 9494, 70])
def test_gemm_bf16_masked_rows_with_8_byte_aligned_row_stride(cuda, N):
    """The vocabulary-layer shape: fp32 output rows of N = 9490 floats (row stride = 2 mod 4) with bias and a row mask —
    the epilogue's shifted 128-bit store path; masked rows must be exactly 0."""
    ops = _ops()
    M, K = 300, 512
    g = torch.Generator().manual_seed(N)
    a = torch.randn(M, K, generator=g)
    b = torch.randn(N, K, generator=g)
    bias = torch.randn(N, generator=g)
    mask = (torch.rand(M, generator=g) > 0.3).to(torch.uint8)
    c = ops.gemm(a.to(cuda), b.to(cuda), bias1=bias.to(cuda), row_mask=mask.to(cuda), precision="bf16")
    ref = (a.bfloat16().double() @ b.bfloat16().double().t() + bias.double()) * mask.double()[:, None]
    H.assert_close_norm(c, ref, 2e-5, "masked tc gemm N=%d" % N)
    assert torch.all(c[mask.to(cuda) == 0] == 0)


@pytest.mark.parametrize("a_mn,b_mn", [(0, 0), (1, 0), (0, 1), (1, 1)])
@pytest.mark.parametrize("M,N,K", [(512, 2048, 2048), (512, 512, 4608), (300, 200, 1000), (128, 64, 64),
                                   (2048, 520, 12288), (96, 9490, 136), (512, 2048, 40000), (1000, 4608, 512),
                                   (640, 9490, 512), (9490, 512, 4096)])
def test_gemm_bf16_operand_majors_tiles_and_split_k(cuda, pair_mode, M, N, K, a_mn, b_mn):
    """Every operand-major combination of the tcgen05 kernel (K-major = rows of K, MN-major = rows of M/N, consumed
    without a transpose), across the BN = 256/128/64 tile plans and the deterministic split-K plans the shapes select
    (per-step contractions with M = batch, weight-gradient contractions with K = tokens); 9490 x 512 x 4096 is the shape
    whose 18-row last m-tile is split off into a second, split-K contraction (150 tiles would need two waves)."""
    ops = _ops()
    g = torch.Generator().manual_seed(M * 7 + N * 3 + K + a_mn * 2 + b_mn)
    a = torch.randn(M, K, generator=g)
    b = torch.randn(N, K, generator=g)
    bias = torch.randn(N, generator=g).to(cuda)
    a_dev = (a.t().contiguous() if a_mn else a).to(cuda)       # MN-major: stored [K][M]
    b_dev = (b.t().contiguous() if b_mn else b).to(cuda)
    kw = dict(M=M, N=N, K=K, bias1=bias, precision="bf16")
    if a_mn:
        kw["a_strides"] = (1, M)
    if b_mn:
        kw["b_strides"] = (1, N)
    c = ops.gemm(a_dev, b_dev, **kw)
    ref = a.bfloat16().double() @ b.bfloat16().double().t() + bias.double().cpu()
    H.assert_close_norm(c, ref, 2e-5, "tc gemm majors (%d,%d) %dx%dx%d" % (a_mn, b_mn, M, N, K))
    c2 = ops.gemm(a_dev, b_dev, **kw)
    assert torch.equal(c, c2), "tensor-core contraction (incl. split-K) must be run-to-run deterministic"


@pytest.mark.gpu
@pytest.mark.parametrize("cluster", ["2,1", "1,2", "2,2", "4,2", "2,4", "4,1", "1,4"])
@pytest.mark.parametrize("a_mn,b_mn", [(0, 0), (1, 0), (0, 1), (1, 1)])
@pytest.mark.parametrize("M,N,K,plan", [(512, 2048, 2048, "64,1"), (512, 4608, 512, "128,1"), (512, 512, 4608, "128,8"),
                                        (512, 2048, 2048, "128,2"), (1000, 4608, 1000, "256,1")])
def test_gemm_bf16_cluster_multicast(cuda, monkeypatch, cluster, M, N, K, plan, a_mn, b_mn):
    """cm x cn thread-block clusters of the multicast contraction: every CTA fetches 1/cn of its A tile and 1/cm of its B tile
    (row slices of K-major tiles, k-row slices of MN-major ones) and TMA-multicasts them along its cluster row / column.
    All operand majors, split-K and non-split plans, bit-identical to the un-clustered kernel (same tiles, same k order)."""
    ops = _ops()
    g = torch.Generator().manual_seed(M + N + K + a_mn * 2 + b_mn)
    a = torch.randn(M, K, generator=g)
    b = torch.randn(N, K, generator=g)
    bias = torch.randn(N, generator=g).to(cuda)
    a_dev = (a.t().contiguous() if a_mn else a).to(cuda)
    b_dev = (b.t().contiguous() if b_mn else b).to(cuda)
    kw = dict(M=M, N=N, K=K, bias1=bias, precision="bf16")
    if a_mn:
        kw["a_strides"] = (1, M)
    if b_mn:
        kw["b_strides"] = (1, N)
    monkeypatch.setenv("ICD_GEMM_FORCE_PLAN", plan)
    monkeypatch.setenv("ICD_GEMM_CLUSTER", "1,1")
    c0 = ops.gemm(a_dev, b_dev, **kw)
    monkeypatch.setenv("ICD_GEMM_CLUSTER", cluster)
    c = ops.gemm(a_dev, b_dev, **kw)
    ref = a.bfloat16().double() @ b.bfloat16().double().t() + bias.double().cpu()
    H.assert_close_norm(c, ref, 2e-5, "clustered tc gemm %s majors (%d,%d) %dx%dx%d" % (cluster, a_mn, b_mn, M, N, K))
    assert torch.equal(c, c0), "cluster multicast must not change a single bit"


@pytest.mark.parametrize("a_mn,b_mn", [(0, 0), (1, 1), (0, 1)])
@pytest.mark.parametrize("M,N,K", [(200, 9490, 512), (64, 300, 2048), (5120, 2048, 520)])
def test_gemm_fp32x3_is_fp32_grade(cuda, M, N, K, a_mn, b_mn):
    """ICD_PREC_FP32X3: fp32 operands split into three bf16 terms, six cross terms summed by one tcgen05 contraction.
    Operand rounding is gone (24 mantissa bits kept); what remains is the tensor core's truncating fp32 accumulator:
    measured ~6e-6 norm-wise at K = 512, i.e. ~70x tighter than single-pass TF32 (4e-4) and ~500x tighter than bf16
    operands (3e-3).  Bound asserted: 2e-5."""
    ops = _ops()
    g = torch.Generator().manual_seed(M + 3 * N + 7 * K)
    a = torch.randn(M, K, generator=g)
    b = torch.randn(N, K, generator=g)
    bias = torch.randn(N, generator=g).to(cuda)
    a_dev = (a.t().contiguous() if a_mn else a).to(cuda)
    b_dev = (b.t().contiguous() if b_mn else b).to(cuda)
    kw = dict(M=M, N=N, K=K, bias1=bias, precision="fp32x3")
    if a_mn:
        kw["a_strides"] = (1, M)
    if b_mn:
        kw["b_strides"] = (1, N)
    c = ops.gemm(a_dev, b_dev, **kw)
    ref = a.double() @ b.double().t() + bias.double().cpu()
    H.assert_close_norm(c, ref, 2e-5, "fp32x3 gemm %dx%dx%d majors (%d,%d)" % (M, N, K, a_mn, b_mn))
    c16 = ops.gemm(a_dev, b_dev, **dict(kw, precision="bf16"))
    assert H.rel_err(c, ref) * 50 < H.rel_err(c16, ref), "fp32x3 must be far tighter than bf16 operands"
    print("fp32x3 rel err %.2e, bf16 rel err %.2e" % (H.rel_err(c, ref), H.rel_err(c16, ref)))


@pytest.mark.gpu
@pytest.mark.parametrize("B,T,P,V", [(5, 7, 196, 300), (64, 24, 196, 9490), (1, 1, 3, 11)])
def test_fused_loss_glue_matches_reference_expression(cuda, B, T, P, V):
    """icd_b200.losses.attention_caption_loss == models/attention.py:401-414 (pack_padded_sequence + CrossEntropyLoss +
    doubly stochastic regulariser), value and gradients w.r.t. the logits and the alphas, in fp64 torch on the CPU."""
    from torch.nn.utils.rnn import pack_padded_sequence
    from icd_b200.losses import attention_caption_loss, alpha_regulariser
    g = torch.Generator().manual_seed(B * 31 + T)
    lens = sorted((int(x) for x in torch.randint(1, T + 1, (B,), generator=g)), reverse=True)
    lens[0] = T
    caps = torch.randint(0, V, (B, T + 1), generator=g)
    preds = torch.randn(B, T, V, generator=g) * 2
    alphas = torch.rand(B, T, P, generator=g) / P
    for b, l in enumerate(lens):                          # the decoder leaves inactive rows at exactly 0
        preds[b, l:] = 0
        alphas[b, l:] = 0
    p64 = preds.double().requires_grad_(True)
    a64 = alphas.double().requires_grad_(True)
    scores = pack_padded_sequence(p64, lens, batch_first=True).data
    targets = pack_padded_sequence(caps[:, 1:], lens, batch_first=True).data
    ref = torch.nn.CrossEntropyLoss()(scores, targets) + ((1.0 - a64.sum(dim=1)) ** 2).mean()
    ref.backward()
    pd = preds.to(cuda).requires_grad_(True)
    ad = alphas.to(cuda).requires_grad_(True)
    loss = attention_caption_loss(pd, caps.to(cuda), lens, ad, alpha_c=1.0)
    (loss * 0.5).backward()                               # a non-trivial upstream gradient, read on the device
    assert abs(loss.item() - ref.item()) < 2e-6 * max(1.0, abs(ref.item()))
    H.assert_close_norm(pd.grad, p64.grad * 0.5, 1e-5, "d_logits")
    H.assert_close_norm(ad.grad, a64.grad * 0.5, 1e-5, "d_alphas")
    reg = alpha_regulariser(alphas.to(cuda), 0.7)
    assert abs(reg.item() - ((0.7 - alphas.double().sum(dim=1)) ** 2).mean().item()) < 1e-6


@pytest.mark.gpu
@pytest.mark.parametrize("B,L,H", [(128, 25, 512), (6, 9, 32), (200, 5, 64), (3, 1, 16), (512, 3, 128)])
def test_persistent_lstm_recurrence_matches_torch(cuda, B, L, H):
    """K8 (csrc/lstm_persistent.cu): the nn.LSTM recurrence of models/baseline.py:106 and its adjoint, each as ONE
    persistent cooperative kernel, against torch autograd over the same recurrence in fp64 (bf16 operands, fp32
    accumulation: stated 5e-3 on the states, 2e-2 on the gate gradients).  Shapes: configs[1], a tiny one (K tail of the
    64-wide k-block, 6 of 128 rows), two / four row tiles, a single step."""
    import helpers as H_                       # (H is the hidden size in this test)
    ops = _ops()
    assert ops.lstm_seq_supported(B, L, H)
    g = torch.Generator().manual_seed(B + L + H)
    w_hh = (torch.rand(4 * H, H, generator=g) * 2 - 1) / H ** 0.5
    xg = torch.randn(L, B, 4 * H, generator=g)
    d_hout = torch.randn(B, L, H, generator=g)
    w64 = w_hh.double().requires_grad_(True)
    x64 = xg.double().requires_grad_(True)
    h = torch.zeros(B, H, dtype=torch.float64)
    c = torch.zeros(B, H, dtype=torch.float64)
    hs, cs = [], []
    for t in range(L):
        gates = h @ w64.t() + x64[t]
        i, f, gg, o = gates.chunk(4, dim=1)
        c = torch.sigmoid(f) * c + torch.sigmoid(i) * torch.tanh(gg)
        h = torch.sigmoid(o) * torch.tanh(c)
        hs.append(h)
        cs.append(c)
    hout64 = torch.stack(hs, dim=1)
    (hout64 * d_hout.double()).sum().backward()
    out = ops.lstm_seq_fwd(w_hh.to(cuda), xg.to(cuda))
    H_.assert_close_norm(out["hout"], hout64, 5e-3, "hout")
    H_.assert_close_norm(out["h_all"][1:], torch.stack(hs, 0), 5e-3, "h_all")
    H_.assert_close_norm(out["c_all"][1:], torch.stack(cs, 0), 5e-3, "c_all")
    assert torch.all(out["h_all"][0] == 0) and torch.all(out["c_all"][0] == 0)
    H_.assert_close_norm(out["hout16"].float().view(B, L, H), out["hout"], 4e-3, "hout16")
    dg, dg16 = ops.lstm_seq_bwd(w_hh.to(cuda), d_hout.to(cuda), out["gates_act"], out["c_all"])
    H_.assert_close_norm(dg, x64.grad, 2e-2, "d gates_pre")            # xg enters the gates additively: d xg == dg
    H_.assert_close_norm(dg16.float().view(L, B, 4 * H), dg, 4e-3, "dg16")
    from icd_b200._lib import lib
    print("lstm_seq backward launch mode:", lib().icd_lstm_seq_bwd_launch_mode())
    assert lib().icd_lstm_seq_bwd_launch_mode() in (1, 2)
    # run-to-run determinism (fixed summation order inside one tcgen05 accumulator)
    out2 = ops.lstm_seq_fwd(w_hh.to(cuda), xg.to(cuda))
    assert torch.equal(out["hout"], out2["hout"]) and torch.equal(out["c_all"], out2["c_all"])


def _ragged_bt(B, T, g, n_empty):
    """Descending decode lengths with dl[0] = T and the last n_empty rows at 0 (Tb = 0) -> (dl, bt)."""
    dl = sorted((int(x) for x in torch.randint(1, T + 1, (B - n_empty,), generator=g)), reverse=True) + [0] * n_empty
    dl[0] = T
    return dl, [sum(1 for l in dl if l > t) for t in range(T)]


PROJ_CASES = {        # B, T, P, A, att_dec row stride, w_full kind, rows with no active step
    "regime_b_like": dict(B=64, T=24, P=196, A=512, ld=512 + 2048 + 2048, w="normal", empty=3),
    "p1": dict(B=7, T=5, P=1, A=64, ld=72, w="normal", empty=2),
    "p28": dict(B=6, T=9, P=28, A=128, ld=128, w="normal", empty=1),
    "p29": dict(B=6, T=9, P=29, A=96, ld=100, w="tiny", empty=1),
    "p57": dict(B=5, T=6, P=57, A=64, ld=68, w="fallback", empty=1),
    "t1_a2048": dict(B=3, T=1, P=29, A=2048, ld=2056, w="normal", empty=0),
    "t104_a512": dict(B=3, T=104, P=29, A=512, ld=512, w="normal", empty=1),
    "t3_a4096_fp32": dict(B=4, T=3, P=30, A=4096, ld=4096, w="normal", empty=1),     # (the bf16 kernels stop at A = 2048)
}


@pytest.mark.parametrize("case", list(PROJ_CASES))
def test_attention_proj_bwd_multi_step_ragged_matches_fp64(cuda, case):
    """The reductions after the time loop over many steps of a ragged batch (one step is covered above):
        d_att_enc, d_w_full, d_b_full, d_b_enc  of  sum_{b, t < Tb, p} d_e[b,t,p] (sum_a relu(att_enc[b,p,a] + att_dec[t,b,a]) w[a] + b_full)
    for icd_attention_proj_bwd (fp32), icd_attention_proj_bwd_bf16 (direct form) and its split form (d_att_dec_all given).
    Edges: pixel tails (P = 1, 29, 57: P % 28 != 0, the clamped loads and the early break), rows with no active step (their
    d_att_enc rows are exactly 0), att_dec_all with a row stride > A (a slice of the decoders' z), exact ties
    att_enc + att_dec == 0 (split form x > -att_dec == direct form x + att_dec > 0), w_full entries from 1e-17 to 1 and one
    below the split form's floor (fallback to the direct form), T = 1 at A = 2048 (1024-thread blocks, two staged rows; these
    failed to launch before the kernels got an instantiation capped at 64 registers), A = 4096 in the fp32 kernel (1024 threads),
    T = 104 at A = 512 (the shared-memory limit; 105 is an argument error).  d_e at inactive (t, b) — and att_dec_all there,
    for the kernels that do not read it in the split form's column dot — is NaN: it must never be read."""
    from icd_b200 import _lib
    ops = _ops()
    c = PROJ_CASES[case]
    B, T, P, A, ld = c["B"], c["T"], c["P"], c["A"], c["ld"]
    g = torch.Generator().manual_seed(B * 1000 + T * 10 + P)
    if case == "regime_b_like":              # bench.py's regime-B lengths, one row in eight, and three rows with no step
        from icd_b200 import synthetic
        _, lens = synthetic.captions(8 * (B - 3), 9490, max_len=25, lengths="ragged")
        dl = [l - 1 for l in lens[::8]] + [0] * 3
        bt = [sum(1 for l in dl if l > t) for t in range(T)]
        assert bt[0] == B - 3 and bt[-1] < bt[12] < bt[0]
    else:
        dl, bt = _ragged_bt(B, T, g, c["empty"])
    active = torch.tensor([[t < dl[b] for t in range(T)] for b in range(B)])           # (B, T)
    att_enc = (torch.randn(B, P, A, generator=g) * 0.5).bfloat16().float()              # exact in both kernels
    dec_buf = torch.randn(T, B, ld, generator=g) * 0.5
    for t in range(T):                       # exact ties: att_dec[t, b, :A/4] = -att_enc[b, p0, :A/4]
        p0 = int(torch.randint(0, P, (1,), generator=g))
        dec_buf[t, :, :A // 4] = -att_enc[:, p0, :A // 4]
    if c["w"] == "normal":
        w = torch.randn(A, generator=g) * 0.2
    else:                                    # magnitudes 1e-17 .. 1, both signs
        w = 10.0 ** (-17 * torch.rand(A, generator=g)) * torch.sign(torch.randn(A, generator=g))
        if c["w"] == "fallback":
            w[A // 3] = 1e-19
    d_e = torch.randn(B, T, P, generator=g)
    # fp64 reference (autograd), one step at a time
    ae64 = att_enc.double().requires_grad_(True)
    w64 = w.double().requires_grad_(True)
    b64 = torch.zeros(1, dtype=torch.float64, requires_grad=True)
    for t in range(T):
        n = bt[t]
        if n == 0:
            continue
        s = torch.relu(ae64[:n] + dec_buf[t, :n, None, :A].double()) @ w64 + b64          # (n, P)
        (s * d_e[:n, t].double()).sum().backward()
    # split-form input: d_att_dec_all[t, b] = w * sum_p [att_enc + att_dec > 0] d_e, 0 at inactive (t, b)
    ddec_buf = torch.zeros(T, B, ld)
    with torch.no_grad():
        for t in range(T):
            n = bt[t]
            m = ((ae64[:n] + dec_buf[t, :n, None, :A].double()) > 0).double()               # (n, P, A)
            ddec_buf[t, :n, :A] = (w64 * (m * d_e[:n, t, :, None].double()).sum(1)).float()
    # never-read entries
    d_e_nan = d_e.clone()
    d_e_nan[~active] = float("nan")
    dec_nan = dec_buf.clone()
    dec_nan[~active.t()] = float("nan")
    dev = lambda x: x.to(cuda)
    dec_nan_d, dec_d, ddec_d = dev(dec_nan)[:, :, :A], dev(dec_buf)[:, :, :A], dev(ddec_buf)[:, :, :A]
    assert dec_nan_d.stride(1) == ld
    want = dict(d_att_enc=ae64.grad, d_w_full=w64.grad, d_b_full=b64.grad, d_b_enc=ae64.grad.sum(dim=(0, 1)))
    empty_rows = [b for b in range(B) if dl[b] == 0]

    def check(res, what):
        d_att_enc, d_wf, d_bf, d_be = res[0], res[-3], res[-2], res[-1]
        H.assert_close_norm(d_att_enc, want["d_att_enc"], 2e-5, what + " d_att_enc")
        H.assert_close_norm(d_wf, want["d_w_full"], 2e-5, what + " d_w_full")
        H.assert_close_norm(d_bf, want["d_b_full"], 1e-4, what + " d_b_full", atol=1e-5)
        H.assert_close_norm(d_be, want["d_b_enc"], 2e-5, what + " d_b_enc")
        if len(res) == 5:
            H.assert_close_norm(res[1].float(), want["d_att_enc"], 4e-3, what + " d_att_enc16")
            assert torch.all(res[1][empty_rows] == 0)
        assert torch.all(d_att_enc[empty_rows] == 0), what + ": rows with no active step"
        assert all(torch.isfinite(x).all() for x in res), what + ": non-finite output (a never-read entry was read)"

    att_enc_d, att_enc16_d, w_d, d_e_d = dev(att_enc), dev(att_enc.bfloat16()), dev(w), dev(d_e_nan)
    check(ops.attention_proj_bwd(att_enc_d, dec_nan_d, w_d, d_e_d, bt), "fp32")
    if case.endswith("_fp32"):
        return
    direct = ops.attention_proj_bwd_bf16(att_enc16_d, dec_nan_d, w_d, d_e_d, bt)
    check(direct, "bf16 direct")
    split = ops.attention_proj_bwd_bf16(att_enc16_d, dec_d, w_d, d_e_d, bt, d_att_dec_all=ddec_d)
    check(split, "bf16 split")
    # the split form's masked sums equal the direct form's bit for bit (exact ties included)
    assert torch.equal(split[0], direct[0]) and torch.equal(split[1], direct[1]) and torch.equal(split[4], direct[4])
    if c["w"] == "fallback":                 # a |w_full| entry below the floor: the direct form, bit for bit
        assert torch.equal(split[2], direct[2])
    if case == "t104_a512":                  # one more step no longer fits the shared memory: an argument error, no launch
        bt1 = bt + [0]
        dec1 = torch.zeros(T + 1, B, A, device=cuda)
        de1 = torch.zeros(B, T + 1, P, device=cuda)
        with pytest.raises(_lib.IcdError):
            ops.attention_proj_bwd(att_enc_d, dec1, w_d, de1, bt1)
        with pytest.raises(_lib.IcdError):
            ops.attention_proj_bwd_bf16(att_enc16_d, dec1, w_d, de1, bt1)


@pytest.mark.parametrize("C,P", [(4, 1), (1028, 50), (2048, 196)])
@pytest.mark.parametrize("T", [1, 31, 32, 33, 65])
@pytest.mark.parametrize("with_mean", [True, False])
def test_attention_enc_grad_multi_step_matches_fp64(cuda, T, C, P, with_mean):
    """icd_attention_enc_grad on its own: d_enc[b,p,c] = sum_{t < Tb} alpha[b,t,p] d_awe[t,b,c] + d_mean[b,c] / P.  The kernel keeps
    d_awe of at most 32 steps in registers and accumulates d_enc in place over the chunks of 32 steps (T = 33, 65); rows with
    Tb = 0 get d_mean / P only (0 without d_mean); C = 4 / 1028: one thread / a partly filled second block of channels.
    alphas and d_awe at inactive (t, b) are NaN: they must never be read."""
    ops = _ops()
    g = torch.Generator().manual_seed(T * 100 + C + P)
    B = 6
    dl, bt = _ragged_bt(B, T, g, 2 if T > 1 else 1)
    alphas = torch.rand(B, T, P, generator=g) / P
    d_awe = torch.randn(T, B, C, generator=g)
    d_mean = torch.randn(B, C, generator=g) if with_mean else None
    ref = torch.zeros(B, P, C, dtype=torch.float64)
    for b in range(B):
        n = dl[b]
        ref[b] = torch.einsum("tp,tc->pc", alphas[b, :n].double(), d_awe[:n, b].double())
        if with_mean:
            ref[b] += d_mean[b].double() / P
    for b in range(B):
        alphas[b, dl[b]:] = float("nan")
        d_awe[dl[b]:, b] = float("nan")
    got = ops.attention_enc_grad(alphas.to(cuda), d_awe.to(cuda), d_mean.to(cuda) if with_mean else None, bt)
    assert torch.isfinite(got).all()
    H.assert_close_norm(got, ref, 1e-5, "d_enc")
    for b in range(B):
        if dl[b] == 0:
            if with_mean:
                H.assert_close_norm(got[b], ref[b], 1e-6, "d_enc of a row with no active step")
            else:
                assert torch.all(got[b] == 0)
        else:
            H.assert_close_norm(got[b], ref[b], 1e-5, "d_enc row %d (%d steps)" % (b, dl[b]))
