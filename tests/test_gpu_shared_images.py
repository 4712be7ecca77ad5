"""GPU tier: captions that share images — ``AttentionDecoder.forward(..., image_index=idx)``.

By definition the result is that of ``forward(encoder_out[idx], ...)`` and the gradient w.r.t. ``encoder_out`` is the sum over
each image's rows.  Every case runs the indexed call and the replicated call in the same tier, and both against fp64 autograd
through oracle/decoders.py on the replicated features:
- fp32 tier: predictions and alphas bit-identical to the replicated call (its weight gradients use split-K atomics, so
  gradients are compared at the DESIGN.md section 3 bars);
- fp32x3 and bf16 (every contraction deterministic), at full size, where K1 runs without split-K at both row counts: forward
  outputs bit-identical, and so are the gradients whose kernels only see per-row data (fc, decode_step, f_beta, dec_att,
  h_lin, c_lin, embedding); everything else (enc_att.*, full_att.*, encoder_out) within the tier's section 3 bars, the tiny
  A = 48 case at the goldens' looser ones;
- run-to-run determinism (torch.equal) of the indexed call in fp32x3 and bf16.
The full-size row schedule is chosen with icd_attention_step_launch_plan_bf16 so that one call visits every bf16 launch form."""
import ctypes
import warnings

import numpy as np
import pytest
import torch

import helpers as H
from oracle import decoders as O

pytestmark = pytest.mark.gpu

ILL = ("attention.enc_att.weight", "attention.enc_att.bias", "attention.dec_att.weight", "attention.dec_att.bias")
PER_ROW = ("fc.", "decode_step.", "f_beta.", "attention.dec_att.", "h_lin.", "c_lin.", "embedding.")
FWD = {"fp32": 1e-4, "fp32x3": 1e-4, "bf16": 5e-3}
GRAD = {"fp32": 1e-3, "fp32x3": 1e-3, "bf16": 1e-2}
GRAD_ILL = {"fp32": 1e-3, "fp32x3": 3e-3, "bf16": 5e-2}
GRAD_ILL_A48 = {"fp32": 1e-3, "fp32x3": 3e-3, "bf16": 1.5e-1}
ENC_GRAD = {"fp32": 1e-3, "fp32x3": 1e-3, "bf16": 3e-2}


def _decoder(cuda, V, A, D, E, precision, dropout=0.0, train=False, wseed=0):
    import icd_b200.models.attention as my_att
    from icd_b200.vocabulary import synthetic_vocab
    case = dict(V=V, A=A, D=D, E=E, dropout=dropout, train=train, wseed=wseed, fine_tune_embedding=True)
    dec = H.build_attention_module(case, my_att.AttentionDecoder, my_att.AttentionDecoderParams, synthetic_vocab(V))
    sd = {k: v.detach().clone() for k, v in dec.state_dict().items()}
    dec = dec.to(cuda)
    dec.precision = precision
    return dec, sd


def _index(counts, seed):
    """Rows of image i = counts[i]; the rows' images in a shuffled order (an image's rows are spread over the batch)."""
    g = np.random.default_rng(seed)
    return torch.from_numpy(g.permutation(np.repeat(np.arange(len(counts)), counts)))


def _masks(dl, D, seed):
    """One (batch_size_t, D) keep-mask per step (what the oracle applies) and the (T, B, D) stack the module takes."""
    g = torch.Generator().manual_seed(seed)
    masks = [(torch.rand(sum(l > t for l in dl), D, generator=g) > 0.5).float() for t in range(max(dl))]
    return masks, H.stack_masks(masks, len(dl), D)


def _run(dec, enc, caps, lens, idx=None, rep=None, mask=None, emb=None, feat_grad=True):
    """forward (indexed by idx, or on the replicated rows enc[rep]) + the reference loss + backward."""
    dec.zero_grad(set_to_none=True)
    dec._dropout_mask_override = mask
    x = enc.detach().clone().requires_grad_(feat_grad)
    if idx is None:
        preds, _, dl, alphas = dec(x[rep.to(x.device)], caps, lens, embeddings=emb)
    else:
        preds, _, dl, alphas = dec(x, caps, lens, embeddings=emb, image_index=idx)
    loss = O.attention_loss(preds, caps, dl, alphas)          # cross-entropy + the alpha regulariser (a d_alphas upstream)
    loss.backward()
    grads = {k: p.grad.detach().clone() for k, p in dec.named_parameters() if p.grad is not None}
    if feat_grad:
        grads["encoder_out"] = x.grad.detach().clone()
    return preds.detach(), alphas.detach(), loss.detach(), grads


def _both(dec, enc, caps, lens, idx, **kw):
    return _run(dec, enc, caps, lens, idx=idx, **kw), _run(dec, enc, caps, lens, rep=idx, **kw)


def _oracle(sd, enc, caps, lens, idx, masks=None, p=0.0, emb=None):
    w = {k: v.double().requires_grad_(True) for k, v in sd.items()}
    e = enc.detach().cpu().double().requires_grad_(True)
    pr, _, dl, al = O.attention_decoder_forward(w, e[idx], caps, lens, dropout_p=p, dropout_masks=masks,
                                                embeddings=None if emb is None else emb.double())
    loss = O.attention_loss(pr, caps, dl, al)
    loss.backward()
    g = {k: v.grad for k, v in w.items() if v.grad is not None}
    g["encoder_out"] = e.grad
    return pr.detach(), al.detach(), g


def _check_bars(what, got, ref, tier, ill, rep=None):
    """got within the tier's bars of ref.  rep (the replicated call, when ref is the fp64 oracle): a gradient beyond its bar
    still passes when the indexed call is as close to fp64 as the call that defines it (a case whose conditioning puts the
    replicated call itself beyond the bar).  Every such pass is reported as a warning, with both errors."""
    preds, alphas, _, grads = got
    rp, ra, rg = ref
    H.assert_close_norm(preds, rp, FWD[tier], "%s predictions" % what)
    H.assert_close_norm(alphas, ra, FWD[tier], "%s alphas" % what)
    assert set(grads) == set(rg), (what, sorted(set(grads) ^ set(rg)))
    for k, g in grads.items():
        r = rg[k].cpu().double()
        if k == "attention.full_att.bias":
            assert float((g.cpu().double() - r).abs().max()) <= 1e-4, what
            continue
        tol = ENC_GRAD[tier] if k == "encoder_out" else (ill[tier] if k in ILL else GRAD[tier])
        err, den = float((g.cpu().double() - r).norm()), float(r.norm())
        if rep is not None and err > tol * den + 1e-7:
            err_rep = float((rep[3][k].cpu().double() - r).norm())
            msg = "%s grad %s: %.3e from fp64, replicated call %.3e, bar %.1e x %.3e" % (what, k, err, err_rep, tol, den)
            assert err <= 1.1 * err_rep + 0.1 * tol * den, msg
            warnings.warn("beyond the section 3 bar, as close to fp64 as the replicated call: " + msg)
            continue
        assert err <= tol * den + 1e-7, "%s grad %s: |a-b| = %.3e > %.1e x %.3e" % (what, k, err, tol, den)


# ------------------------------------------------------------------------------------------------------- tiny dimensions
@pytest.mark.parametrize("tier", ["fp32", "fp32x3", "bf16"])
def test_tiny_train_mode_unsorted_ragged(cuda, tier):
    """The goldens' dimensions (A = 48, D = 32, E = 24, V = 97, C = 2048, P = 196); images with 0, 1, 2, 3 and 7 rows,
    unsorted ragged lengths, train-mode dropout through _dropout_mask_override, the alpha regulariser's d_alphas, and
    encoder_out.requires_grad."""
    counts = [2, 0, 7, 1, 3, 0]
    idx = _index(counts, seed=1)
    B = len(idx)
    lens = [5, 9, 3, 9, 7, 2, 6, 9, 4, 8, 2, 5, 7]
    assert len(lens) == B
    dec, sd = _decoder(cuda, 97, 48, 32, 24, tier, dropout=0.5, train=True, wseed=2)
    enc = H.synthetic.features(len(counts), seed=7)
    caps, _ = H.synthetic.captions(B, 97, max_len=max(lens), seed=8, lengths=lens)
    masks, mask = _masks([l - 1 for l in lens], 32, seed=9)
    ind, rep = _both(dec, enc.to(cuda), caps.to(cuda), lens, idx, mask=mask)
    if tier == "fp32":
        assert torch.equal(ind[0], rep[0]) and torch.equal(ind[1], rep[1])
    assert ind[3]["encoder_out"].shape == enc.shape
    assert float(ind[3]["encoder_out"][1].abs().max()) == 0 and float(ind[3]["encoder_out"][5].abs().max()) == 0
    _check_bars("indexed vs replicated", ind, (rep[0], rep[1], rep[3]), tier, GRAD_ILL_A48)
    _check_bars("indexed vs fp64", ind, _oracle(sd, enc, caps, lens, idx, masks, 0.5), tier, GRAD_ILL_A48, rep=rep)


def test_tiny_bf16_encoder_out_is_consumed_in_place(cuda):
    """A bf16 encoder_out in the bf16 tier (read in place, no fp32 round trip), with its bf16 gradient."""
    counts = [1, 4, 0, 2]
    idx = _index(counts, seed=3)
    lens = [6, 6, 5, 4, 4, 3, 2]
    dec, sd = _decoder(cuda, 97, 48, 32, 24, "bf16", wseed=1)
    enc = H.synthetic.features(len(counts), seed=4).to(torch.bfloat16)
    caps, _ = H.synthetic.captions(len(idx), 97, max_len=6, seed=5, lengths=lens)
    ind, rep = _both(dec, enc.to(cuda), caps.to(cuda), lens, idx)
    assert ind[3]["encoder_out"].dtype == torch.bfloat16 and ind[3]["encoder_out"].shape == enc.shape
    _check_bars("bf16 features, indexed vs replicated", ind, (rep[0], rep[1], rep[3]), "bf16", GRAD_ILL_A48)
    _check_bars("bf16 features, indexed vs fp64", ind, _oracle(sd, enc.float(), caps, lens, idx), "bf16", GRAD_ILL_A48)


@pytest.mark.parametrize("tier", ["fp32", "bf16"])
def test_tiny_precomputed_embeddings(cuda, tier):
    """forward(..., embeddings=) (the use_bert branch) together with an image index."""
    counts = [3, 1, 2]
    idx = _index(counts, seed=6)
    lens = [7, 7, 6, 5, 3, 2]
    dec, sd = _decoder(cuda, 97, 48, 32, 24, tier, wseed=4)
    enc = H.synthetic.features(len(counts), seed=10)
    caps, _ = H.synthetic.captions(len(idx), 97, max_len=7, seed=11, lengths=lens)
    emb = torch.randn(len(idx), 7, 24, generator=torch.Generator().manual_seed(12)) * 0.1
    ind, rep = _both(dec, enc.to(cuda), caps.to(cuda), lens, idx, emb=emb.to(cuda))
    assert "embedding.weight" not in ind[3]
    _check_bars("embeddings, indexed vs replicated", ind, (rep[0], rep[1], rep[3]), tier, GRAD_ILL_A48)
    _check_bars("embeddings, indexed vs fp64", ind, _oracle(sd, enc, caps, lens, idx, emb=emb), tier, GRAD_ILL_A48, rep=rep)


# ------------------------------------------------------------------------------------------------------- full dimensions
V, A, D, E = 9490, 512, 512, 512


@pytest.mark.parametrize("tier", ["fp32", "fp32x3", "bf16"])
def test_full_dimensions_against_fp64(cuda, tier):
    """A = D = E = 512, C = 2048, P = 196, V = 9490 on a few rows (the fp64 oracle stays cheap): unsorted ragged lengths,
    images with 0, 1, 3 and 4 rows."""
    counts = [0, 1, 3, 0, 4]
    idx = _index(counts, seed=13)
    lens = [6, 10, 4, 10, 8, 2, 9, 5]
    dec, sd = _decoder(cuda, V, A, D, E, tier, wseed=0)
    enc = H.synthetic.features(len(counts), seed=14)
    caps, _ = H.synthetic.captions(len(idx), V, max_len=10, seed=15, lengths=lens)
    ind, rep = _both(dec, enc.to(cuda), caps.to(cuda), lens, idx)
    if tier == "fp32":
        assert torch.equal(ind[0], rep[0]) and torch.equal(ind[1], rep[1])
    _check_bars("full dims, indexed vs replicated", ind, (rep[0], rep[1], rep[3]), tier, GRAD_ILL)
    _check_bars("full dims, indexed vs fp64", ind, _oracle(sd, enc, caps, lens, idx), tier, GRAD_ILL, rep=rep)


def _plan(direction, rows):
    from icd_b200 import _lib
    from icd_b200._lib import check
    out = (ctypes.c_int32 * 4)()
    check(_lib.lib().icd_attention_step_launch_plan_bf16(direction, rows, 196, 2048, 512, out), "launch_plan")
    return tuple(out)


def _bwd_form(rows):
    per, shared, grid, deep = _plan(1, rows)
    if shared == 0:
        return "whole rows"
    if shared == rows:
        return "all halves" + (" deep" if deep else "")
    rem = rows % 148                    # the full form splits the rows that fill the last wave, the minimal one the rows beyond it
    return "full balance" if abs(shared - (148 - rem)) <= 1 else "minimal balance"


# batch_size_t per step: every forward and backward launch form of the bf16 attention-step kernels, more than 592 rows first
BT_SCHEDULE = [640, 640, 600, 512, 468, 400, 320, 256, 222, 180, 148, 120, 100, 64, 48, 30, 16, 8, 3, 1]


def _full_case():
    B = BT_SCHEDULE[0]
    dl = [sum(1 for bt in BT_SCHEDULE if bt > r) for r in range(B)]
    lens = [d + 1 for d in dl]
    counts = [i % 8 for i in range(183)]                  # 0 .. 7 rows per image
    counts[-1] += B - sum(counts)
    assert min(counts) == 0 and max(counts) >= 7 and sum(counts) == B
    return _index(counts, seed=21), lens, len(counts)


def test_full_size_schedule_visits_every_launch_form():
    """CPU-side check of the fixture below: its steps hit <= 48, <= 148, <= 222 rows, a minimal-balance count, and more than
    592 rows, forward and backward."""
    idx, lens, n_img = _full_case()
    dl = [l - 1 for l in lens]
    bts = [sum(d > t for d in dl) for t in range(max(dl))]
    assert bts == BT_SCHEDULE
    fwd = {_plan(0, r)[0] * 10 + _plan(0, r)[3] for r in bts}
    assert fwd == {41, 21, 20, 10}                        # 4 per row deep, 2 per row deep / not, whole rows
    bwd = {_bwd_form(r) for r in bts}
    assert {"all halves deep", "all halves", "minimal balance", "full balance"} <= bwd
    assert max(bts) > 4 * 148


@pytest.mark.parametrize("tier", ["fp32", "fp32x3", "bf16"])
def test_full_size_every_launch_form_against_replicated(cuda, tier):
    """640 caption rows over 183 images (0 .. 7 rows each, spread through the batch), lengths that take batch_size_t
    through every bf16 launch form.  Bit-identity where the definition allows it, bars elsewhere, run-to-run determinism."""
    idx, lens, n_img = _full_case()
    dec, _ = _decoder(cuda, V, A, D, E, tier, wseed=0)
    enc = H.synthetic.features(n_img, seed=22).to(cuda)
    caps, _ = H.synthetic.captions(len(idx), V, max_len=max(lens), seed=23, lengths=lens)
    caps = caps.to(cuda)
    ind, rep = _both(dec, enc, caps, lens, idx)
    assert torch.equal(ind[0], rep[0]) and torch.equal(ind[1], rep[1]), "forward outputs differ from the replicated call"
    if tier != "fp32":
        for k, g in ind[3].items():
            if k.startswith(PER_ROW):
                assert torch.equal(g, rep[3][k]), "per-row gradient %s differs from the replicated call" % k
        again = _run(dec, enc, caps, lens, idx=idx)
        assert torch.equal(again[0], ind[0]) and torch.equal(again[1], ind[1])
        for k in ind[3]:
            assert torch.equal(again[3][k], ind[3][k]), "indexed %s not run-to-run deterministic" % k
    _check_bars("640 rows, indexed vs replicated", ind, (rep[0], rep[1], rep[3]), tier, GRAD_ILL)


@pytest.mark.parametrize("tier", ["fp32x3", "bf16"])
def test_full_size_launch_forms_against_fp64_on_sampled_images(cuda, tier):
    """The 640-row launch-form case against fp64 autograd on the rows of five of its images (1, 3, 7, 7 and 9 rows, spread
    over the length-sorted batch, so they run under every forward and backward launch form).  The loss is a fixed random
    projection of predictions and alphas, a sum over rows, so the oracle on those rows alone gives their predictions and
    alphas and the complete feature gradient of the five images."""
    idx, lens, n_img = _full_case()
    dec, sd = _decoder(cuda, V, A, D, E, tier, wseed=0)
    enc = H.synthetic.features(n_img, seed=22)
    caps, _ = H.synthetic.captions(len(idx), V, max_len=max(lens), seed=23, lengths=lens)
    T = max(lens) - 1
    g = torch.Generator().manual_seed(24)
    gp, ga = torch.randn(len(idx), T, V, generator=g), torch.randn(len(idx), T, 196, generator=g)
    x = enc.to(cuda).requires_grad_(True)
    preds, _, dl, alphas = dec(x, caps.to(cuda), lens, image_index=idx)
    ((preds * gp.to(cuda)).sum() + (alphas * ga.to(cuda)).sum()).backward()
    imgs = [1, 3, 7, 15, n_img - 1]
    assert [int((idx == i).sum()) for i in imgs] == [1, 3, 7, 7, 9]
    rows = torch.nonzero(torch.isin(idx, torch.tensor(imgs))).flatten()       # ascending: lengths stay non-increasing
    sub_lens = [lens[r] for r in rows.tolist()]
    Ts = max(sub_lens) - 1
    w = {k: v.double() for k, v in sd.items()}
    e = enc.double().requires_grad_(True)
    pr, _, _, al = O.attention_decoder_forward(w, e[idx[rows]], caps[rows], sub_lens)
    ((pr * gp[rows, :Ts].double()).sum() + (al * ga[rows, :Ts].double()).sum()).backward()
    H.assert_close_norm(preds[rows.to(cuda), :Ts], pr, FWD[tier], "sampled rows: predictions")
    H.assert_close_norm(alphas[rows.to(cuda), :Ts], al, FWD[tier], "sampled rows: alphas")
    H.assert_close_norm(x.grad[imgs], e.grad[imgs], ENC_GRAD[tier], "sampled images: d encoder_out")


def test_data_parallel_sink_equals_plain_backward(cuda):
    """DataParallelClipAdam's overlap mode (the backward writes weight gradients straight into its flat buffer) with an
    image index: the same gradients as the plain backward, bit for bit (bf16 tier, deterministic)."""
    from icd_b200.parallel import DataParallelClipAdam
    counts = [3, 0, 5, 2]
    idx = _index(counts, seed=30)
    lens = [9, 9, 8, 7, 7, 5, 4, 3, 2, 2]
    dec, _ = _decoder(cuda, V, A, D, E, "bf16", wseed=0)
    enc = H.synthetic.features(len(counts), seed=31).to(cuda)
    caps, _ = H.synthetic.captions(len(idx), V, max_len=9, seed=32, lengths=lens)
    caps = caps.to(cuda)
    plain = _run(dec, enc, caps, lens, idx=idx, feat_grad=False)[3]
    opt = DataParallelClipAdam(dec, group=False)
    opt.zero_grad()
    preds, _, dl, alphas = dec(enc, caps, lens, image_index=idx)
    O.attention_loss(preds, caps, dl, alphas).backward()
    assert opt.buf.in_place, "the backward did not write into the flat buffer"
    opt.buf.gather_grads()
    for name, p in zip(opt.buf.names, opt.buf.params):
        off, k = opt.buf.offsets[name]
        assert torch.equal(opt.buf.flat_grad[off:off + k].view_as(p), plain[name]), name
    del dec._icd_grad_sink


def test_bad_index_raises_before_any_launch(cuda):
    from icd_b200._lib import lib
    dec, _ = _decoder(cuda, 97, 48, 32, 24, "bf16")
    enc = H.synthetic.features(3, seed=1).to(cuda)
    caps, lens = H.synthetic.captions(4, 97, max_len=5, seed=2, lengths=[5, 4, 3, 2])
    caps = caps.to(cuda)
    bad = [torch.tensor([0, 1, 2]), torch.tensor([0.0, 1.0, 2.0, 0.0]), torch.tensor([[0, 1, 2, 0]]),
           torch.tensor([0, 1, 3, 0]), torch.tensor([0, -1, 2, 0], device=cuda)]
    for b in bad:
        n0 = lib().icd_launch_count()
        with pytest.raises(ValueError):
            dec(enc, caps, lens, image_index=b)
        assert lib().icd_launch_count() == n0, b


# ------------------------------------------------------------------------------------------------------------------ SCST
def _scst_case(n_img):
    import icd_b200.models.attention as my_att
    from icd_b200.vocabulary import synthetic_vocab
    case = dict(H.BEAM_CASES["beam_small"], dropout=0.5, train=True, fine_tune_embedding=True, end_bias=8.0, emb_scale=1.0)
    dec = H.build_attention_module(case, my_att.AttentionDecoder, my_att.AttentionDecoderParams, synthetic_vocab(case["V"]))
    H.apply_beam_recipe(dec, case)
    return dec, H.synthetic.features(n_img, seed=40), case["V"]


def _reward(seq, ln):
    keep = torch.arange(seq.shape[-1], device=seq.device) < ln[..., None]
    return ((seq.long() * keep).sum(-1) % 11).float() / 11.0


@pytest.mark.parametrize("tier", ["fp32", "bf16"])
def test_scst_matches_the_replicated_computation(cuda, tier):
    """self_critical_loss on the attention decoder (indexed training forward) against the same loss formed by hand on the
    replicated features features[img_idx], from the same samples and advantages."""
    from icd_b200.losses import weighted_token_loss
    from icd_b200.scst import pack_samples, scored_targets, self_critical_loss
    dec, feats, V = _scst_case(6)
    dec = dec.to(cuda)
    dec.precision = tier
    x = feats.to(cuda).requires_grad_(True)
    loss, info = self_critical_loss(dec, x, _reward, 5, V - 3, V - 2, seed=77, max_steps=8)
    loss.backward()
    got = {k: p.grad.clone() for k, p in dec.named_parameters() if p.grad is not None}
    got["features"] = x.grad.clone()
    dec.zero_grad(set_to_none=True)
    pk = pack_samples(dict(seq=info["seq"], len=info["len"]))
    xr = feats.to(cuda).requires_grad_(True)
    dec.eval()
    logits = dec(xr[pk.img_idx], pk.captions, pk.lengths)[0]
    dec.train()
    tgt = scored_targets(pk.captions, pk.lengths, False, getattr(logits, "_icd_row_valid", None))
    w = pk.pack(info["advantages"])[:, None].expand(len(pk.lengths), logits.shape[1]).contiguous()
    ref_loss = weighted_token_loss(logits, tgt, w, info["n_tokens"])
    ref_loss.backward()
    assert abs(float(loss) - float(ref_loss)) <= FWD[tier] * (abs(float(ref_loss)) + 1.0)
    for k, g in got.items():
        r = xr.grad if k == "features" else dict(dec.named_parameters())[k].grad
        if k == "attention.full_att.bias":
            assert float((g - r).abs().max()) <= 1e-5
            continue
        tol = ENC_GRAD[tier] if k == "features" else (GRAD_ILL_A48[tier] if k in ILL else GRAD[tier])
        H.assert_close_norm(g, r, tol, "scst %s grad %s" % (tier, k), atol=1e-9)


def test_scst_peak_memory_drops_by_the_replicated_features(cuda):
    """64 images x m = 5: the indexed training step allocates at least 80 % of R * P * C * 4 bytes less at its peak than
    the same step on features[img_idx]."""
    from icd_b200.scst import pack_samples, self_critical_loss
    n, m = 64, 5
    dec, feats, V = _scst_case(n)
    dec = dec.to(cuda)
    dec.precision = "bf16"
    x = feats.to(cuda)
    with torch.no_grad():
        _, info = self_critical_loss(dec, x, _reward, m, V - 3, V - 2, seed=5, max_steps=8)
    pk = pack_samples(dict(seq=info["seq"], len=info["len"]))
    dec.eval()

    def peak(indexed):
        dec.zero_grad(set_to_none=True)
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats()
        base = torch.cuda.memory_allocated()
        if indexed:
            preds, _, dl, al = dec(x, pk.captions, pk.lengths, image_index=pk.img_idx_host)
        else:
            preds, _, dl, al = dec(x[pk.img_idx], pk.captions, pk.lengths)
        O.attention_loss(preds, pk.captions, dl, al).backward()
        del preds, al
        torch.cuda.synchronize()
        return torch.cuda.max_memory_allocated() - base

    peak(True)                                            # warm-up: first-use allocations of both paths
    peak(False)
    p_ind, p_rep = peak(True), peak(False)
    R, P, C = n * m, 196, 2048
    print("peak allocated: indexed %.1f MB, replicated %.1f MB, R*P*C*4 = %.1f MB" % (p_ind / 1e6, p_rep / 1e6, R * P * C * 4 / 1e6))
    assert p_rep - p_ind >= 0.8 * R * P * C * 4
