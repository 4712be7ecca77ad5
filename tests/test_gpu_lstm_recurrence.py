"""Step-local parity of the persistent LSTM recurrence (K8, csrc/lstm_persistent.cu) against an fp64 restatement of the
same operation fed with the kernel's own operands (tests/lstm_recurrence_reference.py), plus its shape rules.

The whole-tensor comparison of test_gpu_ops.py::test_persistent_lstm_recurrence_matches_torch carries errors through the
recurrence and so needs 5e-3; here every step is checked on its own against a per-element bound derived from the kernel's
arithmetic, block by block in the kernel's work split, so one wrong weight column, one stale row tile or one dropped
k-block at one step fails and is named.
"""
import ctypes

import pytest
import torch

import helpers as H_
import lstm_recurrence_reference as R


def _lib():
    from icd_b200._lib import lib
    return lib()


# ---------------------------------------------------------------------------------------------------------------------
# CPU tier
# ---------------------------------------------------------------------------------------------------------------------
def test_lstm_seq_shape_rules_without_a_device():
    """icd_lstm_seq_shape_ok: H % 16 == 0, H / 4 <= 148, 1 <= B <= 512, L >= 1 — answered without a device."""
    ok = _lib().icd_lstm_seq_shape_ok
    for H in (16, 48, 80, 512, 528, 592):
        for B in (1, 127, 128, 129, 385, 512):
            assert ok(B, 1, H) == 1, (B, H)
            assert ok(B, 200, H) == 1, (B, H)
    for H in (0, 8, 24, 40, 100, 520, 600, 608, 1024):           # not whole 16-unit groups, or more than 148 forward CTAs
        assert ok(128, 25, H) == 0, H
    for B in (0, -1, 513, 640, 1024):                            # more than 4 row tiles of 128
        assert ok(B, 25, 512) == 0, B
    for L in (0, -3):
        assert ok(128, L, 512) == 0, L


def _whole_tensor_criterion(w_hh, xg, sim):
    """The whole-tensor criterion of test_persistent_lstm_recurrence_matches_torch (fp64 recurrence on the unrounded
    weights, 5e-3 norm-wise on hout, h_all, c_all) -> True if it accepts."""
    L, B, H4 = xg.shape
    H = H4 // 4
    w64, x64 = w_hh.double(), xg.double()
    h = torch.zeros(B, H, dtype=torch.float64)
    c = torch.zeros(B, H, dtype=torch.float64)
    hs, cs = [], []
    for t in range(L):
        i, f, g, o = (h @ w64.t() + x64[t]).chunk(4, dim=1)
        c = torch.sigmoid(f) * c + torch.sigmoid(i) * torch.tanh(g)
        h = torch.sigmoid(o) * torch.tanh(c)
        hs.append(h)
        cs.append(c)
    try:
        H_.assert_close_norm(sim["hout"], torch.stack(hs, dim=1), 5e-3, "hout")
        H_.assert_close_norm(sim["h_all"][1:], torch.stack(hs, 0), 5e-3, "h_all")
        H_.assert_close_norm(sim["c_all"][1:], torch.stack(cs, 0), 5e-3, "c_all")
    except AssertionError:
        return False
    return True


def test_block_criterion_catches_what_the_whole_tensor_bound_misses():
    """A CPU simulation of the forward kernel (fp32 from bf16 operands) passes the block criterion; three localised faults
    at one step are each rejected, and the failure names the faulty block:
      * one CTA contracting with its neighbour's W_hh columns,
      * one row tile reading h from the step before,
      * one CTA's row tile with its K-tail k-block (k >= 64) dropped.
    The whole-tensor 5e-3 criterion accepts at least one of them."""
    B, L, H = 200, 25, 80                                        # 2 row tiles (the second partial), 20 CTAs, a 16-wide K tail
    g = torch.Generator().manual_seed(7)
    w_hh = (torch.rand(4 * H, H, generator=g) * 2 - 1) / H ** 0.5
    xg = torch.randn(L, B, 4 * H, generator=g)
    t0, cta, tile = L - 1, 5, 1
    cols = torch.cat([torch.arange(gt * H + 4 * cta, gt * H + 4 * cta + 4) for gt in range(4)])
    rows = slice(tile * R.BM, B)

    def neighbour_columns(t, A, W):
        if t != t0:
            return None
        Wc = W.clone()
        Wc[cols] = W[cols + 4]
        return A @ Wc.t()

    def stale_h(t, A, W):
        if t != t0:
            return None
        pre = A @ W.t()
        pre[rows] = 0.0 if t == 0 else sim_ok["h16"][(t - 1) * B:t * B].float()[rows] @ W.t()
        return pre

    def k_tail_dropped(t, A, W):
        if t != t0:
            return None
        pre = A @ W.t()
        A2 = A.clone()
        A2[:, 64:] = 0
        pre[rows, cols] = (A2 @ W.t())[rows][:, cols]
        return pre

    sim_ok = R.simulate_forward(w_hh, xg)
    fails, worst = R.check_forward(w_hh, xg, sim_ok["h16"], sim_ok["c_all"], sim_ok["gates_act"], sim_ok["h_all"])
    assert not fails, fails
    assert worst < 1.0
    accepted = []
    for name, fault in (("neighbour columns", neighbour_columns), ("stale h", stale_h), ("K tail", k_tail_dropped)):
        sim = R.simulate_forward(w_hh, xg, fault)
        fails, worst = R.check_forward(w_hh, xg, sim["h16"], sim["c_all"], sim["gates_act"], sim["h_all"])
        print("%-18s block criterion: %d messages, worst %.3g x the bound; whole-tensor 5e-3: %s"
              % (name, len(fails), worst, "accepts" if _whole_tensor_criterion(w_hh, xg, sim) else "rejects"))
        assert fails, name
        assert all("step %d" % t0 in m for m in fails if "..." not in m), (name, fails)
        if name != "stale h":
            assert all("CTA %d " % cta in m for m in fails if "..." not in m), (name, fails)
        if _whole_tensor_criterion(w_hh, xg, sim):
            accepted.append(name)
    assert accepted, "the whole-tensor criterion rejected every fault: the comparison no longer shows what it should"


# ---------------------------------------------------------------------------------------------------------------------
# GPU tier
# ---------------------------------------------------------------------------------------------------------------------
def _largest_admitted_h(B):
    return max(h for h in range(16, 4 * 148 + 1, 16) if _lib().icd_lstm_seq_supported(B, 1, h))


def _padded(shape, dtype, dev, fill=float("nan")):
    """A buffer of ``shape`` filled with ``fill``, followed by one sentinel row of its last dimension."""
    n = 1
    for s in shape:
        n *= s
    buf = torch.full((n + shape[-1],), fill, dtype=dtype, device=dev)
    buf[n:] = torch.arange(shape[-1], device=dev).to(dtype) * -0.5 - 3.0
    return buf, buf[:n].view(*shape), buf[n:].clone()


# (B, H, L): 1 .. 4 row tiles with partial last tiles, K tails (H = 16, 48, 80: one partial k-block; 528: 8 full + one
# of 16), more than 128 CTAs (528, the largest admitted H), one step, two steps, long recurrences
CASES = [
    (1, 16, 1), (127, 48, 25), (128, 80, 2), (129, 512, 25), (300, 528, 25), (385, 80, 200), (512, 512, 25),
    (512, 16, 200), (128, 512, 200), (129, 48, 1), (128, "max", 25), (512, "max", 25), (300, "max", 2),
]


@pytest.mark.gpu
@pytest.mark.parametrize("B,H,L", CASES)
def test_persistent_recurrence_step_local_parity(cuda, B, H, L):
    """Forward: for every step t, pre = h16[t] bf16(W_hh)^T + xg[t] in fp64 on the kernel's h16 rows, the activations and
    c = f c_all[t] + i g, h = o tanh(c) on the kernel's c_all[t] -> gates_act[t], c_all[t+1], h_all[t+1] within the
    per-element bound of one step; hout[:, t] == h_all[t+1], h16[t+1] == bf16(h_all[t+1]), hout16 == bf16(hout) bit for bit.
    Backward: dh_t = d_hout[:, t] + dg16[t+1] bf16(W_hh) on the kernel's dg16, the cell adjoint on the kernel's gates and
    cell states with the dc carry in fp64 -> dg[t] within its bound; dg16 == bf16(dg) bit for bit.
    Every output starts as NaN (written through the C ABI, not the allocating wrappers); a sentinel row after each buffer
    must be untouched."""
    if H == "max":
        H = _largest_admitted_h(B)
    L_ = _lib()
    assert L_.icd_lstm_seq_supported(B, L, H), "B=%d L=%d H=%d refused by the persistent predicate" % (B, L, H)
    g = torch.Generator().manual_seed(B * 1000 + H + L)
    w_hh = ((torch.rand(4 * H, H, generator=g) * 2 - 1) / H ** 0.5).to(cuda)
    xg = torch.randn(L, B, 4 * H, generator=g).to(cuda)
    d_hout = torch.randn(B, L, H, generator=g).to(cuda)
    f32, b16 = torch.float32, torch.bfloat16
    bufs = {}
    for name, shape, dt in (("gates_act", (L, B, 4 * H), f32), ("c_all", (L + 1, B, H), f32), ("h_all", (L + 1, B, H), f32),
                            ("hout", (B, L, H), f32), ("h16", ((L + 1) * B, H), b16), ("hout16", (B * L, H), b16),
                            ("dg", (L, B, 4 * H), f32), ("dg16", (L * B, 4 * H), b16), ("dc", (B, H), f32)):
        bufs[name] = _padded(shape, dt, cuda)
    o = {k: v[1] for k, v in bufs.items()}
    bar = torch.zeros(64, device=cuda, dtype=torch.int32)
    p = lambda t: ctypes.c_void_p(t.data_ptr())                  # noqa: E731
    from icd_b200._lib import check, stream_ptr
    n0 = L_.icd_launch_count()
    check(L_.icd_lstm_seq_fwd(B, L, H, p(w_hh), p(xg), p(o["gates_act"]), p(o["c_all"]), p(o["h_all"]), p(o["hout"]),
                              p(o["h16"]), p(o["hout16"]), p(bar), stream_ptr()), "icd_lstm_seq_fwd")
    check(L_.icd_lstm_seq_bwd(B, L, H, p(w_hh), p(d_hout), p(o["gates_act"]), p(o["c_all"]), p(o["dc"]), p(o["dg"]),
                              p(o["dg16"]), p(bar), stream_ptr()), "icd_lstm_seq_bwd")
    torch.cuda.synchronize()
    assert L_.icd_launch_count() - n0 == 2                       # one persistent kernel per direction
    assert L_.icd_lstm_seq_bwd_launch_mode() == 1, "the backward was not launched cooperatively"
    for name, (buf, view, sentinel) in bufs.items():
        assert torch.equal(buf[view.numel():], sentinel), "%s: the row after the buffer was written" % name
        if name != "dc":
            assert not torch.isnan(view).any(), "%s: %d elements never written" % (name, int(torch.isnan(view).sum()))
    assert torch.all(o["h_all"][0] == 0) and torch.all(o["c_all"][0] == 0)
    assert torch.equal(o["hout"], o["h_all"][1:].permute(1, 0, 2))
    assert torch.equal(o["h16"].view(L + 1, B, H)[1:], o["h_all"][1:].to(b16))
    assert torch.equal(o["hout16"], o["hout"].reshape(B * L, H).to(b16))
    assert torch.equal(o["dg16"], o["dg"].reshape(L * B, 4 * H).to(b16))

    fails, worst_f = R.check_forward(w_hh, xg, o["h16"], o["c_all"], o["gates_act"], o["h_all"])
    fails_b, worst_b = R.check_backward(w_hh, d_hout, o["gates_act"], o["c_all"], o["dg"], o["dg16"])
    print("B=%d H=%d L=%d: largest error / bound  forward %.3g  backward %.3g" % (B, H, L, worst_f, worst_b))
    assert not fails + fails_b, "\n".join(fails + fails_b)
