"""GPU tier: self-critical sequence training (icd_b200.scst.self_critical_loss, losses.weighted_token_loss) and the weighted
cross-entropy gradient kernels under it (icd_weighted_cross_entropy_bwd / _fwd_grad16).

- Kernel level: both entry points against the fp64 closed form w_r * scale * (softmax - onehot), every output written, and
  bit-identical to the unweighted kernels when every weight is 1.
- Decoder level: both decoders on samples of the real sampler, every gradient against fp64 autograd through the oracle
  (tests/scst_reference.py states the loss), in the fp32, fp32x3 and bf16 tiers.
- The forward's logp against the sampler's, greedy limits, determinism, refusals, and a small learning run per decoder."""
import ctypes

import pytest
import torch

import helpers as Hh
import scst_reference as SC
from oracle import decoders as O
from test_gpu_baseline_beam import CASES as BASE_CASES, build_decoder, image_features

pytestmark = pytest.mark.gpu

MAX_STEPS = 8
M = 5
SEED = 0x5C57
ILL_CONDITIONED = ("attention.enc_att.weight", "attention.enc_att.bias", "attention.dec_att.weight",
                   "attention.dec_att.bias")
# DESIGN.md section 3 bars (norm-wise, per gradient tensor); the tiny A = 48 attention case takes the bf16 goldens' 1.5e-1 on
# the four ill-conditioned attention-projection gradients, the baseline bf16 tier the 2e-2 of test_gpu_baseline_parity.py
GRAD = {"fp32": 1e-3, "fp32x3": 1e-3, "bf16": 1e-2}
GRAD_ILL = {"fp32": 1e-3, "fp32x3": 3e-3, "bf16": 1.5e-1}
GRAD_BASE_BF16 = 2e-2
# bf16 training tier: bar on the largest |forward logp - sampler logp| over the scored tokens (the test prints the gap).
# Measured on a B200: 2.1e-2 (attention case), 5.5e-3 (baseline case); the fp32 and fp32x3 tiers: <= 3.9e-5.
BF16_LOGP_GAP = 5e-2


# ------------------------------------------------------------------------------------------------------------ kernel level
def _ce_call(weighted, fused, logits, targets, inv_count, weights=None, upstream=None, want32=True):
    """Run one cross-entropy gradient entry point on NaN-filled outputs (bf16 pad columns included)."""
    from icd_b200 import _lib
    from icd_b200._lib import ptr, stream_ptr
    L = _lib.lib()
    R, V = logits.shape
    ld16 = (V + 7) // 8 * 8
    dev = logits.device
    d16 = torch.full((R, ld16), float("nan"), device=dev, dtype=torch.bfloat16)
    if fused:
        rl = torch.full((R,), float("nan"), device=dev)
        lse = torch.full((R,), float("nan"), device=dev)
        args = [ctypes.c_int64(R), V, ptr(logits), ptr(targets), ctypes.c_float(inv_count)]
        args += [ptr(weights)] if weighted else []
        args += [ptr(rl), ptr(lse), ptr(d16), ctypes.c_int64(ld16), stream_ptr()]
        fn = L.icd_weighted_cross_entropy_fwd_grad16 if weighted else L.icd_cross_entropy_fwd_grad16
        assert fn(*args) == 0, L.icd_last_error_string()
        return None, d16, rl, lse
    from icd_b200 import ops
    _, lse = ops.cross_entropy_fwd(logits, targets)
    d32 = torch.full((R, V), float("nan"), device=dev) if want32 else None
    args = [ctypes.c_int64(R), V, ptr(logits), ptr(targets), ptr(lse), ptr(upstream), ctypes.c_float(inv_count)]
    args += [ptr(weights)] if weighted else []
    args += [ptr(d32), ptr(d16), ctypes.c_int64(ld16), stream_ptr()]
    fn = L.icd_weighted_cross_entropy_bwd if weighted else L.icd_cross_entropy_bwd
    assert fn(*args) == 0, L.icd_last_error_string()
    return d32, d16, None, lse


def _logits(R, V, cuda, seed):
    g = torch.Generator(device=cuda).manual_seed(seed)
    x = torch.randn(R, V, device=cuda, generator=g) * 3.0
    t = torch.randint(0, V, (R,), device=cuda, generator=g)
    t[::7] = -1                                                           # ignored rows
    w = torch.randn(R, device=cuda, generator=g)
    w[1::11] = 0.0
    w[2::11] = 1e20
    w[3::11] = -1e-20
    w[4::11] = -3.5
    return x, t, w


def _closed_form(x, t, w, scale):
    """fp64 reference and the per-element bound: exp(x - lse) in fp32 carries the rounding of lse and of x - lse (each scaled
    by |x - lse| or |lse| in the exponent) and ~2 ulps of the exponential; then the products — all in fp32 ulps."""
    x64 = x.double()
    lse = torch.logsumexp(x64, dim=1, keepdim=True)
    p = torch.exp(x64 - lse)
    oh = torch.zeros_like(p)
    valid = t >= 0
    oh[valid, t[valid]] = 1.0
    ws = (w.double() * scale)[:, None]
    ref = ws * (p - oh)
    ref[~valid] = 0.0
    u = 2.0 ** -23
    bound = ws.abs() * (u * p * (8.0 + 2.0 * (x64 - lse).abs() + 2.0 * lse.abs()) + 2 * u * oh) + 1e-44
    bound[~valid] = 0.0
    return ref, bound


@pytest.mark.parametrize("R,V", [(12288, 9490), (333, 131), (64, 7)])
@pytest.mark.parametrize("fused", [False, True])
def test_weighted_kernels_against_the_closed_form(cuda, R, V, fused):
    x, t, w = _logits(R, V, cuda, R + V)
    inv = 1.0 / 1234.0
    up = torch.tensor([0.75], device=cuda)
    d32, d16, rl, _ = _ce_call(True, fused, x, t, inv, weights=w, upstream=up)
    ref, bound = _closed_form(x, t, w, inv * (1.0 if fused else 0.75))
    if d32 is not None:
        assert not torch.isnan(d32).any()
        err = (d32.double() - ref).abs()
        assert bool((err <= bound).all()), "fp32: worst %.3e of its bound" % float((err / bound.clamp_min(1e-300)).max())
    assert not torch.isnan(d16.float()).any(), "an entry of the bf16 gradient (pad columns included) was not written"
    assert bool((d16[:, V:].float() == 0).all())
    err16 = (d16[:, :V].double() - ref).abs()
    bound16 = bound + 2.0 ** -8 * ref.abs()
    assert bool((err16 <= bound16).all()), "bf16: worst %.3e of its bound" % float((err16 / bound16.clamp_min(1e-300)).max())
    zero_rows = (w == 0) | (t < 0)
    assert bool((d16[zero_rows].float() == 0).all())
    if rl is not None:                                                   # the one-pass kernel's loss stays unweighted
        _, _, rl0, _ = _ce_call(False, True, x, t, inv)
        assert torch.equal(rl, rl0)


@pytest.mark.parametrize("R,V", [(12288, 9490), (333, 131)])
def test_unit_weights_reproduce_the_unweighted_kernels(cuda, R, V):
    x, t, _ = _logits(R, V, cuda, 7 * R + V)
    one = torch.ones(R, device=cuda)
    up = torch.tensor([0.3], device=cuda)
    inv = 1.0 / 977.0
    a32, a16, _, _ = _ce_call(False, False, x, t, inv, upstream=up)
    b32, b16, _, _ = _ce_call(True, False, x, t, inv, weights=one, upstream=up)
    assert torch.equal(a32, b32) and torch.equal(a16, b16)
    _, a16, arl, alse = _ce_call(False, True, x, t, inv)
    _, b16, brl, blse = _ce_call(True, True, x, t, inv, weights=one)
    assert torch.equal(a16, b16) and torch.equal(arl, brl) and torch.equal(alse, blse)


# ------------------------------------------------------------------------------------------------------------ decoders
# The decoder-level cases keep the default initialisation of the embeddings (emb_scale 1), as the goldens on which the bars of
# DESIGN.md section 3 were set do.  The beam fixtures' x30 embeddings saturate the LSTM gates, where sigma'(z) carries a
# relative error of about |z| * 2^-8 from bf16 operands, far above those bars.  <end> is made likely enough (end_bias) that
# the samples of a case end at several lengths and some are truncated at MAX_STEPS.
def _attention(end_bias=8.0, n_img=4):
    import icd_b200.models.attention as my_att
    from icd_b200.vocabulary import synthetic_vocab
    case = dict(Hh.BEAM_CASES["beam_small"], dropout=0.5, train=True, fine_tune_embedding=True, end_bias=end_bias,
                emb_scale=1.0)
    dec = Hh.build_attention_module(case, my_att.AttentionDecoder, my_att.AttentionDecoderParams, synthetic_vocab(case["V"]))
    Hh.apply_beam_recipe(dec, case)
    return dec, Hh.beam_features(case)[:n_img], case["V"]


def _baseline(n_img=6):
    case = dict(BASE_CASES["small"], end_bias=2.0, n_img=n_img, emb_scale=1.0)
    return build_decoder(case), image_features(case), case["V"]


def make(kind):
    return _attention() if kind == "attention" else _baseline()


def token_hash_reward(seq, ln):
    """A deterministic reward with signed advantages against either baseline."""
    S = seq.shape[-1]
    keep = torch.arange(S, device=seq.device) < ln[..., None]
    return ((seq.long() * keep).sum(-1) % 11).float() / 11.0


def word_fraction(target, end_id):
    """The fraction of a caption's words (tokens after <start>, <end> excluded) equal to ``target``."""
    def fn(seq, ln):
        t = torch.arange(seq.shape[-1], device=seq.device)
        word = (t >= 1) & (t < ln[..., None]) & (seq != end_id)
        return (word & (seq == target)).sum(-1).float() / word.sum(-1).clamp_min(1).float()
    return fn


def _run(dec, feats, V, cuda, reward=token_hash_reward, want_feat=False, **kw):
    from icd_b200.scst import self_critical_loss
    dec.zero_grad(set_to_none=True)
    x = feats.to(cuda).clone().requires_grad_(want_feat)
    kw = dict(dict(n_samples=M, seed=SEED, max_steps=MAX_STEPS), **kw)
    loss, info = self_critical_loss(dec, x, reward, start_id=V - 3, end_id=V - 2, **kw)
    loss.backward()
    grads = {k: p.grad.detach().clone() for k, p in dec.named_parameters() if p.grad is not None}
    if want_feat:
        grads["features"] = x.grad.detach().clone()
    return loss.detach(), info, grads


def _oracle(dec, feats, info, base, want_feat):
    """fp64 gradients of the SCST loss, and of the same loss with |A| (the scale of the terms a signed gradient sums)."""
    from icd_b200.scst import pack_samples, scored_targets
    pk = pack_samples(dict(seq=info["seq"].cpu(), len=info["len"].cpu()))
    w = {k: v.detach().cpu().double().requires_grad_(True) for k, v in dec.state_dict().items()}
    f = feats.double().requires_grad_(want_feat)
    x = f[pk.img_idx]
    logits = (O.baseline_decoder_forward(w, x, pk.captions) if base else
              O.attention_decoder_forward(w, x, pk.captions, pk.lengths)[0])
    tgt = scored_targets(pk.captions, pk.lengths, base)
    adv = pk.pack(info["advantages"].cpu().double())
    names = list(w) + (["features"] if want_feat else [])
    leaves = list(w.values()) + ([f] if want_feat else [])
    out = {}
    for tag, a in (("signed", adv), ("abs", adv.abs())):
        lo = SC.loss(logits, tgt, a)
        out[tag] = dict(zip(names, torch.autograd.grad(lo, leaves, retain_graph=True, allow_unused=True)))
        out[tag + "_loss"] = float(lo)
    return out


TIERS = [("attention", "fp32", False), ("attention", "fp32x3", True), ("attention", "bf16", False),
         ("baseline", "fp32", True), ("baseline", "fp32x3", False), ("baseline", "bf16", True)]


@pytest.mark.parametrize("kind,tier,want_feat", TIERS)
def test_gradients_against_fp64(cuda, kind, tier, want_feat):
    """Signed advantages can make a gradient small against its terms, so each gradient's error is judged against the larger
    of its own fp64 norm and the fp64 gradient norm of sum |A| * CE / N."""
    dec, feats, V = make(kind)
    dec = dec.to(cuda)
    dec.precision = tier
    loss, info, grads = _run(dec, feats, V, cuda, want_feat=want_feat)
    ln, ended = info["len"].cpu(), info["ended"].cpu()
    assert 0 < int(ended.sum()) < ended.numel() and len(set(ln.flatten().tolist())) >= 3, \
        "the case needs samples of several lengths, some truncated"
    adv = info["advantages"]
    assert bool((adv > 0).any()) and bool((adv < 0).any())
    assert dec.training, "the previous module mode is restored"
    ref = _oracle(dec, feats, info, kind == "baseline", want_feat)
    assert abs(float(loss) - ref["signed_loss"]) <= 1e-3 * ref["abs_loss"] + 1e-7
    seen = 0
    for k, g in grads.items():
        r, ra = ref["signed"][k], ref["abs"][k]
        if k == "attention.full_att.bias":
            assert float(g.abs().max()) <= 1e-5
            continue
        tol = GRAD_ILL[tier] if k in ILL_CONDITIONED else GRAD[tier]
        if kind == "baseline" and tier == "bf16":
            tol = GRAD_BASE_BF16
        den = max(float(r.norm()), float(ra.norm()))
        err = float((g.cpu().double() - r).norm())
        assert err <= tol * den, "%s %s %s: |g - fp64| = %.3e > %.1e * %.3e" % (kind, tier, k, err, tol, den)
        seen += 1
    want = sum(1 for _, p in dec.named_parameters() if p.requires_grad) + int(want_feat)
    assert len(grads) == want and seen >= want - 1


def test_bf16_grad_only_is_bit_identical(cuda):
    dec, feats, V = make("attention")
    dec = dec.to(cuda)
    dec.precision = "bf16"
    la, _, ga = _run(dec, feats, V, cuda)
    lb, _, gb = _run(dec, feats, V, cuda, bf16_grad_only=True)
    assert torch.equal(la, lb)
    for k in ga:
        assert torch.equal(ga[k], gb[k]), k


@pytest.mark.parametrize("kind", ["attention", "baseline"])
@pytest.mark.parametrize("tier", ["fp32", "fp32x3", "bf16"])
def test_forward_logp_is_the_samplers(cuda, kind, tier):
    from icd_b200.gen_captions import sample_captions
    dec, feats, V = make(kind)
    dec = dec.to(cuda)
    dec.precision = tier
    _, info, _ = _run(dec, feats, V, cuda)
    with torch.no_grad():
        s = sample_captions(dec, feats.to(cuda), M, V - 3, V - 2, seed=SEED, max_steps=MAX_STEPS, want_logp=True)
    assert torch.equal(s["seq"], info["seq"]) and torch.equal(s["len"], info["len"])
    gap = float((info["logp"] - s["logp"]).abs().max())
    print("%s %s: max |forward logp - sampler logp| = %.3e" % (kind, tier, gap))
    assert gap <= (1e-4 if tier != "bf16" else BF16_LOGP_GAP), gap


@pytest.mark.parametrize("kind", ["attention", "baseline"])
def test_greedy_samples_have_zero_advantage_loss_and_gradient(cuda, kind):
    dec, feats, V = make(kind)
    dec = dec.to(cuda)
    loss, info, grads = _run(dec, feats, V, cuda, temperature=0.0, want_feat=True)
    assert int((info["advantages"] != 0).sum()) == 0
    assert float(loss) == 0.0
    for k, g in grads.items():
        assert int(torch.count_nonzero(g)) == 0, k


@pytest.mark.parametrize("kind", ["attention", "baseline"])
def test_determinism_and_returned_seed(cuda, kind):
    dec, feats, V = make(kind)
    dec = dec.to(cuda)
    dec.precision = "fp32x3"
    la, ia, ga = _run(dec, feats, V, cuda, baseline="mean")
    lb, ib, gb = _run(dec, feats, V, cuda, baseline="mean")
    assert torch.equal(la, lb)
    for k in ga:
        assert torch.equal(ga[k], gb[k]), k
    torch.manual_seed(123)
    lc, ic, gc = _run(dec, feats, V, cuda, seed=None)
    ld, idd, gd = _run(dec, feats, V, cuda, seed=ic["seed"])
    assert torch.equal(ic["seq"], idd["seq"]) and torch.equal(lc, ld)
    for k in gc:
        assert torch.equal(gc[k], gd[k]), k


def test_refusals_raise_before_the_training_forward(cuda):
    from icd_b200 import ops
    from icd_b200.gen_captions import sample_captions
    dec, feats, V = make("baseline")
    dec = dec.to(cuda)
    x = feats.to(cuda)
    n0 = ops.launch_count()
    with pytest.raises(ValueError):
        _run(dec, feats, V, cuda, sample_precision="bf16")
    assert ops.launch_count() == n0
    with torch.no_grad():
        sample_captions(dec, x, M, V - 3, V - 2, seed=SEED, max_steps=MAX_STEPS, want_logp=True)
    sampler_launches = ops.launch_count() - n0
    bad = [lambda s, l: torch.zeros(s.shape[0], M + 1, device=s.device),
           lambda s, l: torch.full(l.shape, float("nan"), device=s.device),
           lambda s, l: torch.zeros(l.shape, device="cpu")]
    for fn in bad:
        n1 = ops.launch_count()
        with pytest.raises(ValueError):
            _run(dec, feats, V, cuda, reward=fn)
        assert ops.launch_count() - n1 == sampler_launches, "only the sampler ran"


def _learn(cuda, kind, steps, lr, target):
    """``steps`` seeded SCST steps (leave-one-out baseline, Adam) with the word-fraction reward of ``target`` -> the held-out
    mean reward (8 samples per image at a seed no step uses) before and after."""
    from icd_b200.gen_captions import sample_captions
    dec, feats, V = _attention(n_img=8) if kind == "attention" else _baseline(n_img=32)
    dec = dec.to(cuda)
    dec.precision = "fp32x3"
    reward = word_fraction(target, V - 2)
    x = feats.to(cuda)

    def held_out():
        with torch.no_grad():
            s = sample_captions(dec, x, 8, V - 3, V - 2, seed=987654321, max_steps=MAX_STEPS)
        return float(reward(s["seq"], s["len"]).mean())

    before = held_out()
    opt = torch.optim.Adam([p for p in dec.parameters() if p.requires_grad], lr=lr)
    for k in range(steps):
        _run(dec, feats, V, cuda, reward=reward, seed=1000 + k, baseline="mean")
        opt.step()
    return before, held_out()


# Deterministic at fixed seeds.  Measured on a B200 (held-out mean reward before -> after): attention 0.021 -> 0.646, baseline
# 0.013 -> 0.850; the margins ask for about half of those rises.
LEARN = {"attention": dict(steps=30, lr=1e-2, target=7, margin=0.3),
         "baseline": dict(steps=30, lr=1e-2, target=7, margin=0.4)}


@pytest.mark.parametrize("kind", ["attention", "baseline"])
def test_scst_raises_the_reward(cuda, kind):
    cfg = LEARN[kind]
    before, after = _learn(cuda, kind, cfg["steps"], cfg["lr"], cfg["target"])
    print("%s: held-out mean reward %.4f -> %.4f" % (kind, before, after))
    assert after - before >= cfg["margin"], (before, after)
