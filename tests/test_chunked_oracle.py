"""CPU tier: the row-chunked fp64 oracle (tests/helpers.oracle_fp64_chunked, the checker of the timed-configuration and
regime-B parity tests) equals the one-shot oracle — loss and every parameter gradient, and its opt-in per-step and per-row
outputs — for equal and for ragged (descending) lengths, with a train-mode dropout keep-mask.  And the per-step / per-row
criteria of tests/test_gpu_ragged_regime_b.py catch the localised errors they are there for, which the norm-wise bounds
over whole tensors let through."""
import pytest
import torch

import helpers as H
from oracle import decoders as O


def _case(lengths, B=10, max_len=9):
    import icd_b200.models.attention as my_att
    from icd_b200.vocabulary import synthetic_vocab
    case = dict(B=B, V=61, A=16, D=8, E=12, max_len=max_len, lengths=lengths or [max_len] * B, wseed=3, iseed=5, dropout=0.5,
                train=True, fine_tune_embedding=False)
    dec = H.build_attention_module(case, my_att.AttentionDecoder, my_att.AttentionDecoderParams,
                                   synthetic_vocab(case["V"]))
    sd = dec.state_dict()
    enc, caps, lens = H.att_inputs(case)
    dl = [l - 1 for l in lens]
    T = max(dl)
    keep = H.seeded_keep_mask(T, case["B"], case["D"], 0.5, seed=9)
    return case, sd, enc, caps, lens, dl, keep


def _one_shot(sd, enc, caps, lens, dl, keep):
    """The one-shot oracle: predictions, alphas, loss, parameter gradients and the gradient w.r.t. encoder_out."""
    T = max(dl)
    w = {k: v.detach().double().clone().requires_grad_(k != "embedding.weight") for k, v in sd.items()}
    e64 = enc.double().requires_grad_(True)
    masks = [keep[t, :sum(1 for l in dl if l > t)].double() for t in range(T)]
    p, _, d, a = O.attention_decoder_forward(w, e64, caps, lens, dropout_p=0.5, dropout_masks=masks)
    loss = O.attention_loss(p, caps, d, a)
    loss.backward()
    return p.detach(), a.detach(), loss, w, e64.grad


@pytest.mark.parametrize("lengths", [None, [9, 9, 8, 8, 6, 5, 3, 2, 2, 1]])
def test_chunked_oracle_equals_one_shot(lengths):
    case, sd, enc, caps, lens, dl, keep = _case(lengths)
    p, a, loss, w, d_enc = _one_shot(sd, enc, caps, lens, dl, keep)
    T = max(dl)
    g = torch.Generator().manual_seed(1)
    cand_p = (p * (1 + 1e-3 * torch.randn(p.shape, generator=g, dtype=torch.float64))).float()
    cand_a = (a * (1 + 1e-3 * torch.randn(a.shape, generator=g, dtype=torch.float64))).float()
    cand_e = (d_enc * (1 + 1e-3 * torch.randn(d_enc.shape, generator=g, dtype=torch.float64))).float()
    r = H.oracle_fp64_chunked(sd, enc, caps, lens, keep_mask=keep, p=0.5, frozen=("embedding.weight",), chunk=3,
                              cuda_preds=p.float(), cuda_alphas=a.float())
    assert abs(r["loss"] - loss.item()) < 1e-12 * abs(loss.item())
    assert set(r["grads"]) == {k for k, v in w.items() if v.grad is not None}
    for k, gr in r["grads"].items():
        H.assert_close_norm(gr, w[k].grad, 1e-11, k, atol=1e-15)      # full_att.bias: true value 0, only noise
    assert r["err"]["predictions"] < 1e-6 and r["err"]["alphas"] < 1e-6
    assert "step_sums" not in r and "row_sums" not in r              # opt-in outputs only on request
    # opt-in outputs, two candidates: per-step sums of predictions / alphas, per-row sums of d encoder_out
    r2 = H.oracle_fp64_chunked(sd, enc, caps, lens, keep_mask=keep, p=0.5, frozen=("embedding.weight",), chunk=3,
                               cuda_preds={"x": p.float(), "y": cand_p}, cuda_alphas={"x": a.float(), "y": cand_a},
                               per_step=True, cuda_d_enc={"x": d_enc.float(), "y": cand_e})
    assert r2["loss"] == r["loss"] and all(torch.equal(r2["grads"][k], r["grads"][k]) for k in r["grads"])
    for cand, (cp, ca, ce) in {"x": (p.float(), a.float(), d_enc.float()), "y": (cand_p, cand_a, cand_e)}.items():
        for name, ref, got in (("predictions", p, cp), ("alphas", a, ca)):
            want = torch.stack([((got[:, t].double() - ref[:, t]) ** 2).sum(dim=(0, 1)) for t in range(T)], 0)
            want_ref = torch.stack([(ref[:, t] ** 2).sum() for t in range(T)], 0)
            s = r2["step_sums"][cand][name]
            assert s.shape == (T, 2)
            assert torch.allclose(s[:, 0], want, rtol=1e-6, atol=1e-30) and torch.allclose(s[:, 1], want_ref, rtol=1e-12)
            assert abs(H.aggregate_rel_err(s) - r2["err"][cand][name]) < 1e-6 * r2["err"][cand][name] + 1e-15
        rows = r2["row_sums"][cand]
        de = ce.double().reshape(case["B"], -1) - d_enc.reshape(case["B"], -1)
        assert torch.allclose(rows[:, 0], (de ** 2).sum(dim=1), rtol=1e-6, atol=1e-30)
        assert torch.allclose(rows[:, 1], (d_enc.reshape(case["B"], -1) ** 2).sum(dim=1), rtol=1e-9)
    re = H.row_rel_err(r2["row_sums"]["y"])
    live = torch.tensor(dl) > 0                   # (a row of length 1 has no step: reference and candidate 0, error 0)
    assert float(re.max()) < 2e-3 and float(re[live].min()) > 5e-4 and torch.all(re[~live] == 0)
    # the single-candidate form returns the sums without the candidate level
    r3 = H.oracle_fp64_chunked(sd, enc, caps, lens, keep_mask=keep, p=0.5, frozen=("embedding.weight",), chunk=4,
                               cuda_preds=cand_p, cuda_alphas=cand_a, per_step=True, cuda_d_enc=cand_e)
    assert torch.allclose(r3["step_sums"]["alphas"], r2["step_sums"]["y"]["alphas"], rtol=1e-9, atol=1e-30)
    assert torch.allclose(r3["row_sums"], r2["row_sums"]["y"], rtol=1e-9, atol=1e-30)


def test_per_step_and_per_row_criteria_catch_what_the_norm_wise_bounds_miss():
    """Resolution of the regime-B criteria (bf16-tier bounds of tests/test_gpu_ragged_regime_b.py) on a ragged batch whose
    last step has two of 32 rows: the one-shot oracle's outputs plus bf16-sized noise pass every criterion; three localised
    corruptions — the alphas of the last step's rows, d encoder_out of one row x 1.03, the predictions of the rows that leave
    the batch after step t — each pass the norm-wise bound over the whole tensor and are each rejected by the per-step or the
    per-row criterion."""
    import test_gpu_ragged_regime_b as RB
    lengths = [9] * 2 + [8] * 6 + [7] * 6 + [6] * 5 + [5] * 5 + [4] * 4 + [3] * 2 + [2] * 2
    case, sd, enc, caps, lens, dl, keep = _case(lengths, B=32)
    p, a, _, _, d_enc = _one_shot(sd, enc, caps, lens, dl, keep)
    T, B = max(dl), len(dl)
    bt = [sum(1 for l in dl if l > t) for t in range(T)]
    assert bt[-1] == 2 and bt[-2] == 8
    g = torch.Generator().manual_seed(2)
    noisy = lambda x, e: x * (1 + e * torch.randn(x.shape, generator=g, dtype=torch.float64))
    base = dict(p=noisy(p, 1e-3), a=noisy(a, 1e-3), e=noisy(d_enc, RB.ROW_BOUND["bf16"] / 8))
    bad_alphas = dict(base, a=base["a"].clone())
    bad_alphas["a"][:bt[-1], T - 1] *= 1.02                           # the last step's rows
    bad_row = dict(base, e=base["e"].clone())
    bad_row["e"][20] *= 1.03                                          # one row of d encoder_out
    bad_leavers = dict(base, p=base["p"].clone())
    bad_leavers["p"][bt[T - 1]:bt[T - 2], T - 2] *= 1.02              # the rows whose last step is T - 2
    cands = dict(clean=base, alphas=bad_alphas, row=bad_row, leavers=bad_leavers)
    r = H.oracle_fp64_chunked(sd, enc, caps, lens, keep_mask=keep, p=0.5, frozen=("embedding.weight",), chunk=8,
                              cuda_preds={k: c["p"].float() for k, c in cands.items()},
                              cuda_alphas={k: c["a"].float() for k, c in cands.items()}, per_step=True,
                              cuda_d_enc={k: c["e"].float() for k, c in cands.items()})
    b = RB._bounds("bf16")

    def verdict(k):
        agg = (r["err"][k]["predictions"] < b["out"] and r["err"][k]["alphas"] < b["out"]
               and H.aggregate_rel_err(r["row_sums"][k]) < b["grad"])
        steps = all(float(H.step_rel_err(r["step_sums"][k][n]).max()) < b["out"] for n in ("predictions", "alphas"))
        rows = not H.row_spread_failures(H.row_rel_err(r["row_sums"][k]), b["row"], RB.ROW_K)
        return agg, steps, rows
    assert verdict("clean") == (True, True, True)
    assert verdict("alphas") == (True, False, True)
    assert verdict("row") == (True, True, False)
    assert verdict("leavers") == (True, False, True)
