"""CPU tier: self-critical sequence training (icd_b200.scst) against its restatement (tests/scst_reference.py) — packing of
sampler outputs, scored targets, the two baselines — and, for a tiny decoder of each kind, the packed training forward of the
fp64 oracle against the fp64 sampling reference; then the weighted cross-entropy entry points' argument refusals through the
built library (no GPU needed)."""
import ctypes

import pytest
import torch

import helpers as Hh
import sampling_reference as SR
import scst_reference as SC
from oracle import decoders as O
from test_sampling_reference import _small_baseline


def _hand_made():
    """3 images x 3 samples, max_steps = 6 (S = 8): length ties, truncated samples (len 8) and junk beyond each length."""
    ln = torch.tensor([[4, 8, 4], [2, 4, 8], [8, 3, 4]], dtype=torch.int32)
    g = torch.Generator().manual_seed(3)
    seq = torch.randint(1, 50, (3, 3, 8), generator=g, dtype=torch.int32)
    seq[..., 0] = 97
    return dict(seq=seq, len=ln)


def test_packing_of_a_hand_made_sampler_output():
    from icd_b200.scst import pack_samples, scored_targets
    s = _hand_made()
    pk = pack_samples(s)
    ref = SC.pack(s["seq"].tolist(), s["len"].tolist())
    assert pk.perm.tolist() == [1, 5, 6, 0, 2, 4, 8, 7, 3] == ref["perm"]        # stable: ties keep i*m + j
    assert pk.lengths == [8, 8, 8, 4, 4, 4, 4, 3, 2] == ref["lengths"]
    assert pk.img_idx.tolist() == [0, 1, 2, 0, 0, 1, 2, 2, 1] == ref["img_idx"]
    assert pk.captions.dtype == torch.int64 and torch.equal(pk.captions, ref["captions"])
    assert pk.captions[8, 2:].eq(0).all() and pk.captions[8, :2].tolist() == s["seq"][1, 0, :2].tolist()
    for base in (False, True):
        tgt = scored_targets(pk.captions, pk.lengths, base)
        assert torch.equal(tgt, SC.targets(ref["captions"], ref["lengths"], base)), base
        assert int((tgt >= 0).sum()) == sum(pk.lengths) - len(pk.lengths)
    # row 8 is image 1, sample 0 (len 2): one scored token, <start> -> seq[1, 0, 1]
    assert scored_targets(pk.captions, pk.lengths, False)[8].tolist() == [int(s["seq"][1, 0, 1])] + [-1] * 6
    assert scored_targets(pk.captions, pk.lengths, True)[8].tolist() == [-1, int(s["seq"][1, 0, 1])] + [-1] * 6
    x = torch.randn(3, 3, 5, generator=torch.Generator().manual_seed(1))
    assert torch.equal(pk.unpack(pk.pack(x)), x)
    assert torch.equal(pk.pack(x)[0], x[0, 1])


def test_baselines_and_advantages():
    from icd_b200.scst import baseline_rewards
    r = torch.rand(4, 5, generator=torch.Generator().manual_seed(2))
    greedy = torch.rand(4, generator=torch.Generator().manual_seed(3))
    assert torch.equal(baseline_rewards(r, "greedy", greedy), SC.baseline_rewards(r, "greedy", greedy))
    b = baseline_rewards(r, "mean")
    assert torch.allclose(b, SC.baseline_rewards(r, "mean"), atol=1e-6, rtol=0)
    assert torch.allclose((r - b).sum(dim=1), torch.zeros(4), atol=1e-5)      # leave-one-out advantages sum to 0 per image
    with pytest.raises(ValueError):
        baseline_rewards(r[:, :1], "mean")


def test_mean_baseline_with_one_sample_raises():
    from icd_b200.scst import self_critical_loss
    dec = _small_baseline_module()
    with pytest.raises(ValueError):
        self_critical_loss(dec, torch.zeros(2, 24), lambda s, l: None, 1, 128, 129, baseline="mean")
    with pytest.raises(ValueError):
        self_critical_loss(dec, torch.zeros(2, 24), lambda s, l: None, 2, 128, 129, sample_precision="bf16")


def _small_baseline_module():
    import icd_b200.models.baseline as my_base
    p = my_base.BaselineDecoderParams()
    p.hidden_size, p.embed_size, p.vocab_size = 32, 24, 131
    return my_base.BaselineDecoder(p)


def _attention_case():
    import icd_b200.models.attention as my_att
    from icd_b200.vocabulary import synthetic_vocab
    case = dict(Hh.BEAM_CASES["beam_small"], dropout=0.0, train=False, fine_tune_embedding=True, end_bias=6.0)
    dec = Hh.build_attention_module(case, my_att.AttentionDecoder, my_att.AttentionDecoderParams, synthetic_vocab(case["V"]))
    Hh.apply_beam_recipe(dec, case)
    w = {k: v.detach().double() for k, v in dec.state_dict().items()}
    return w, Hh.beam_features(case)[:3].double(), case["V"]


@pytest.mark.parametrize("kind", ["baseline", "attention"])
def test_packed_forward_scores_the_sampled_tokens(kind):
    """Draw in fp64 with the sampling reference, pack, run the fp64 oracle's training forward on the packed captions: -CE at
    every scored (r, t) is the reference sampler's logp at the same (image, sample, step)."""
    from icd_b200.scst import pack_samples, scored_targets
    base = kind == "baseline"
    if base:
        w, feats, V = _small_baseline()
        feats = feats[:4]
        w["linear.bias"] = w["linear.bias"].clone()
        w["linear.bias"][V - 2] = 2.0                           # <end> likely enough for lengths 2 .. 8 at max_steps 6
        start = SR.baseline_start
    else:
        w, feats, V = _attention_case()
        start = SR.attention_start
    m, max_steps = 3, 6
    S = max_steps + 2
    n = feats.shape[0]
    seq = torch.zeros(n, m, S, dtype=torch.int32)
    ln = torch.zeros(n, m, dtype=torch.int32)
    logp = torch.zeros(n, m, max_steps + 1, dtype=torch.float64)
    for i in range(n):
        step, st = start(w, feats[i] if base else feats[i:i + 1])
        for j, smp in enumerate(SR.sample_image(step, st, m, V - 3, V - 2, max_steps, 1.0, 0, 0xABCDEF, i)):
            seq[i, j, :smp["len"]] = torch.tensor(smp["seq"], dtype=torch.int32)
            ln[i, j] = smp["len"]
            logp[i, j, :smp["len"] - 1] = torch.tensor(smp["logp"], dtype=torch.float64)
    assert len(set(ln.flatten().tolist())) >= 2 and int((ln == S).sum()) >= 1, "the case needs ragged and truncated samples"
    pk = pack_samples(dict(seq=seq, len=ln))
    x = feats[pk.img_idx]
    if base:
        logits = O.baseline_decoder_forward(w, x, pk.captions)
    else:
        logits = O.attention_decoder_forward(w, x, pk.captions, pk.lengths)[0]
    tgt = scored_targets(pk.captions, pk.lengths, base)
    lp = torch.log_softmax(logits, dim=2)
    n_scored = 0
    for r in range(len(pk.lengths)):
        i, j = int(pk.perm[r]) // m, int(pk.perm[r]) % m
        for t in range(tgt.shape[1]):
            if tgt[r, t] < 0:
                continue
            s = SC.step_of(t, base)
            assert int(tgt[r, t]) == int(seq[i, j, s])
            assert abs(float(lp[r, t, tgt[r, t]]) - float(logp[i, j, s - 1])) <= 1e-12, (r, t)
            n_scored += 1
    assert n_scored == int((ln - 1).sum())
    # the loss definition over the packed rows: -(1/N) sum A * logp
    adv = torch.randn(n, m, dtype=torch.float64, generator=torch.Generator().manual_seed(4))
    want = -(adv[:, :, None] * logp).sum() / n_scored
    assert abs(float(SC.loss(logits, tgt, pk.pack(adv))) - float(want)) <= 1e-12 * max(1.0, abs(float(want)))


# ------------------------------------------------------------------------------------------------------------ C ABI
def _bwd(L, R=4, V=131, weights=256, d16=256, ld16=136):
    f = ctypes.c_void_p
    return L.icd_weighted_cross_entropy_bwd(ctypes.c_int64(R), V, f(256), f(256), f(256), f(256), ctypes.c_float(0.5),
                                            f(weights) if weights else None, f(256), f(d16) if d16 else None,
                                            ctypes.c_int64(ld16), None)


def _fg16(L, R=4, V=131, weights=256, ld16=136):
    f = ctypes.c_void_p
    return L.icd_weighted_cross_entropy_fwd_grad16(ctypes.c_int64(R), V, f(256), f(256), ctypes.c_float(0.5),
                                                   f(weights) if weights else None, f(256), f(256), f(256),
                                                   ctypes.c_int64(ld16), None)


@pytest.mark.parametrize("which", ["bwd", "fwd_grad16"])
def test_weighted_cross_entropy_refusals(which):
    from icd_b200 import _lib
    L = _lib.lib()
    call = _bwd if which == "bwd" else _fg16
    assert call(L, weights=0) < 0 and b"weights" in L.icd_last_error_string()
    assert call(L, ld16=132) < 0 and b"ld16" in L.icd_last_error_string()
    assert call(L, ld16=128) < 0 and b"ld16" in L.icd_last_error_string()            # shorter than V
    if which == "fwd_grad16":
        assert call(L, V=60000, ld16=60000) < 0 and b"shared memory" in L.icd_last_error_string()
    assert _lib.DEFINES["ICD_B200_ABI_VERSION"] == 18
    assert "icd_weighted_cross_entropy_bwd" in _lib.FUNCTIONS and "icd_weighted_cross_entropy_fwd_grad16" in _lib.FUNCTIONS
