"""Step-local fp64 restatement of the persistent LSTM recurrence (csrc/lstm_persistent.cu), with a per-element error bound
derived from the kernel's arithmetic, evaluated block by block in the kernel's own work split.

Every step is recomputed from the kernel's OWN operands of that step (its bf16 h_{t-1} rows, its saved gates and cell
states, its bf16 dg_{t+1} rows), so errors are not carried from step to step and the bound is that of one step:

  contraction  fp32 accumulation of exact bf16 x bf16 products over K terms, in any order, each addition rounded at
               most one ulp (truncation included): |err| <= K 2^-23 sum_k |a_k w_k|; the epilogue additions likewise;
  sigmoidf_    1 / (1 + expf(-x)): expf is within 2 ulp (CUDA C Programming Guide, mathematical functions), the add
               and the IEEE division one rounding each: |err| <= sigma'(x) |dx| + 8u sigma;
  tanhf        within 2 ulp: |err| <= (1 - tanh^2) |dx| + 4u |tanh|   (+ the smallest normal, for results near 0);
  products, sums and 1 - x^2 of values carrying an error: first-order propagation plus one rounding per operation,
               bounded by the same expression evaluated on magnitudes.
u = 2^-24 is the unit roundoff of fp32.  The bound is a worst case; the largest observed error is reported as a fraction
of it (measured fractions: profiles/r04_baseline_parity.md).

Blocks: forward, (step, 128-row tile, CTA = 4 hidden units, all four gates); backward, (step, 128-row tile, cluster = 16
hidden units).  A failure names the block.
"""
import torch

U = 2.0 ** -24
TINY = 2.0 ** -126
BM = 128


def bf16(x):
    """Round to bf16 (round-to-nearest-even, as __float2bfloat16_rn) and return as fp64."""
    return x.to(torch.bfloat16).to(torch.float64)


def _sig(x):
    return torch.sigmoid(x)


def forward_reference(w_hh, xg, h16, c_all):
    """fp64 step-local forward from the kernel's operands.
    w_hh (4H,H) fp32, xg (L,B,4H) fp32, h16 ((L+1)B,H) bf16 [the kernel's], c_all (L+1,B,H) fp32 [the kernel's]
    -> dict of references and bounds: gates (L,B,4H), c (L,B,H) = c_{t+1}, h (L,B,H) = h_{t+1}, each with '<name>_bound'."""
    L, B, H4 = xg.shape
    H = H4 // 4
    W = bf16(w_hh)                                               # (4H, H)
    A = h16.to(torch.float64).view(L + 1, B, H)[:L]             # step t reads h_t (row block t)
    x = xg.double()
    pre = A @ W.t() + x                                          # (L, B, 4H)
    S = A.abs() @ W.abs().t()
    e_pre = 2 * U * ((H + 2) * S + 2 * x.abs())
    i, f, g, o = pre.split(H, dim=2)
    ei, ef, eg, eo = e_pre.split(H, dim=2)
    si, sf, so = _sig(i), _sig(f), _sig(o)
    tg = torch.tanh(g)
    d_si = si * (1 - si) * ei + 8 * U * si
    d_sf = sf * (1 - sf) * ef + 8 * U * sf
    d_so = so * (1 - so) * eo + 8 * U * so
    d_tg = (1 - tg * tg) * eg + 4 * U * tg.abs() + TINY
    cp = c_all.double()[:L]
    c = sf * cp + si * tg
    d_c = cp.abs() * d_sf + tg.abs() * d_si + si * d_tg + d_si * d_tg + 3 * U * (sf * cp.abs() + si * tg.abs())
    tc = torch.tanh(c)
    d_tc = (1 - tc * tc) * d_c + 4 * U * tc.abs() + TINY
    h = so * tc
    d_h = tc.abs() * d_so + so * d_tc + d_so * d_tc + 2 * U * (so * tc.abs())
    return dict(gates=torch.cat([si, sf, tg, so], dim=2), gates_bound=torch.cat([d_si, d_sf, d_tg, d_so], dim=2),
                c=c, c_bound=d_c, h=h, h_bound=d_h)


def backward_reference(w_hh, d_hout, gates_act, c_all, dg16):
    """fp64 step-local backward from the kernel's operands: dh_t = d_hout[:, t] + dg16_{t+1} bf16(W_hh), the cell adjoint on
    the kernel's saved gates / cell states, the dc carry kept in fp64 (its bound is carried along: |f| e + one rounding).
    -> dict(dg (L,B,4H), dg_bound)"""
    L, B, H4 = gates_act.shape
    H = H4 // 4
    W = bf16(w_hh)                                               # (4H, H): dh = dg W
    G = dg16.to(torch.float64).view(L, B, 4 * H)
    dho = d_hout.double().permute(1, 0, 2)                       # (L, B, H)
    dhh = torch.zeros(L, B, H, dtype=torch.float64, device=G.device)
    Sb = torch.zeros_like(dhh)
    if L > 1:
        dhh[:L - 1] = G[1:] @ W
        Sb[:L - 1] = G[1:].abs() @ W.abs()
    dh = dhh + dho
    e_dh = 2 * U * ((H + 5) * Sb + dho.abs())                    # four K = H partial sums, summed in rank order, + d_hout
    ga = gates_act.double()
    cs = c_all.double()
    dg = torch.empty(L, B, 4 * H, dtype=torch.float64, device=G.device)
    bound = torch.empty_like(dg)
    dc = torch.zeros(B, H, dtype=torch.float64, device=G.device)
    e_dc = torch.zeros_like(dc)
    for t in range(L - 1, -1, -1):
        i, f, g, o = ga[t].split(H, dim=1)
        cp, cn = cs[t], cs[t + 1]
        d, ed = dh[t], e_dh[t]
        tc = torch.tanh(cn)
        etc = 4 * U * tc.abs() + TINY
        one_m = 1 - tc * tc
        e_one_m = 2 * tc.abs() * etc + 2 * U * (1 + tc * tc)
        d_o = d * tc
        e_do = tc.abs() * ed + d.abs() * etc + U * d_o.abs()
        dcx = dc + d * o * one_m
        e_dcx = e_dc + o * one_m * ed + (d * o).abs() * e_one_m + 3 * U * (dc.abs() + (d * o).abs() * (1 + tc * tc))
        d_i, d_g, d_f = dcx * g, dcx * i, dcx * cp
        pi = d_i * i * (1 - i)
        pf = d_f * f * (1 - f)
        pg = d_g * (1 - g * g)
        po = d_o * o * (1 - o)
        e_pi = g.abs() * i * (1 - i) * e_dcx + 4 * U * (dcx * g).abs() * i * (1 + i)
        e_pf = cp.abs() * f * (1 - f) * e_dcx + 4 * U * (dcx * cp).abs() * f * (1 + f)
        e_pg = i * (1 - g * g) * e_dcx + 4 * U * (dcx * i).abs() * (1 + g * g)
        e_po = o * (1 - o) * e_do + 4 * U * d_o.abs() * o * (1 + o)
        dg[t] = torch.cat([pi, pf, pg, po], dim=1)
        bound[t] = torch.cat([e_pi, e_pf, e_pg, e_po], dim=1) + TINY
        dc = dcx * f
        e_dc = f * e_dcx + U * dc.abs()
    return dict(dg=dg, dg_bound=bound)


def block_ratios(got, ref, bound, units_per_block, gates):
    """max over each block of |got - ref| / bound (NaN -> inf).  got/ref/bound (L, B, gates*H) -> (L, MT, H / units_per_block)."""
    L, B, N = ref.shape
    H = N // gates
    r = (got.double().to(ref.device) - ref).abs() / bound
    r = torch.where(torch.isnan(r), torch.full_like(r, float("inf")), r)
    MT = (B + BM - 1) // BM
    pad = torch.zeros(L, MT * BM, N, dtype=r.dtype, device=r.device)
    pad[:, :B] = r
    return pad.view(L, MT, BM, gates, H // units_per_block, units_per_block).amax(dim=(2, 3, 5)).cpu()


def block_failures(ratios, what, unit_name, units_per_block, limit=1.0):
    """-> list of messages naming the blocks whose worst element exceeds the bound."""
    bad = (ratios > limit).nonzero().tolist()
    msgs = []
    for t, mt, c in bad[:8]:
        msgs.append("%s: step %d, rows %d..%d, %s %d (units %d..%d): %.3g x the bound"
                    % (what, t, mt * BM, mt * BM + BM - 1, unit_name, c, c * units_per_block,
                       (c + 1) * units_per_block - 1, float(ratios[t, mt, c])))
    if len(bad) > 8:
        msgs.append("%s: ... %d blocks over the bound in all" % (what, len(bad)))
    return msgs


def check_forward(w_hh, xg, h16, c_all, gates_act, h_all):
    """Forward block criterion -> (failure messages, largest error / bound over all outputs)."""
    ref = forward_reference(w_hh, xg, h16, c_all)
    fails, worst = [], 0.0
    for name, got, gates in (("gates_act", gates_act, 4), ("c_all", c_all[1:], 1), ("h_all", h_all[1:], 1)):
        key = {"gates_act": "gates", "c_all": "c", "h_all": "h"}[name]
        r = block_ratios(got, ref[key], ref[key + "_bound"], 4, gates)
        fails += block_failures(r, name, "CTA", 4)
        worst = max(worst, float(r.max()))
    return fails, worst


def check_backward(w_hh, d_hout, gates_act, c_all, dg, dg16):
    """Backward block criterion -> (failure messages, largest error / bound)."""
    ref = backward_reference(w_hh, d_hout, gates_act, c_all, dg16)
    r = block_ratios(dg, ref["dg"], ref["dg_bound"], 16, 4)
    return block_failures(r, "dg", "cluster", 16), float(r.max())


def simulate_forward(w_hh, xg, corrupt=None):
    """The forward recurrence as the kernel computes it, in fp32 from bf16 operands (CPU; the accumulation order differs
    from the tensor core's, which the bound covers).  corrupt(t, A, W) -> pre-activations (B, 4H) fp32 or None lets a test
    inject a fault at one step.  -> dict(gates_act, c_all, h_all, h16) in the kernel's layouts."""
    L, B, H4 = xg.shape
    H = H4 // 4
    W = w_hh.to(torch.bfloat16).float()
    h16 = torch.zeros((L + 1) * B, H, dtype=torch.bfloat16)
    c_all = torch.zeros(L + 1, B, H)
    h_all = torch.zeros(L + 1, B, H)
    gates = torch.empty(L, B, 4 * H)
    for t in range(L):
        A = h16[t * B:(t + 1) * B].float()
        pre = corrupt(t, A, W) if corrupt is not None else None
        if pre is None:
            pre = A @ W.t()
        pre = pre + xg[t]
        i, f, g, o = pre.split(H, dim=1)
        i, f, g, o = torch.sigmoid(i), torch.sigmoid(f), torch.tanh(g), torch.sigmoid(o)
        c = f * c_all[t] + i * g
        h = o * torch.tanh(c)
        gates[t] = torch.cat([i, f, g, o], dim=1)
        c_all[t + 1] = c
        h_all[t + 1] = h
        h16[(t + 1) * B:(t + 2) * B] = h.to(torch.bfloat16)
    return dict(gates_act=gates, c_all=c_all, h_all=h_all, h16=h16, hout=h_all[1:].permute(1, 0, 2).contiguous())
