"""GPU tier: beam search over the BaselineDecoder (icd_baseline_beam_search, gen_captions.baseline_beam_search_batched)
against its definition (tests/baseline_beam_reference.py), against itself (compaction, chunking, run-to-run) and
against the training forward of the same module."""
import functools

import pytest
import torch
import torch.nn.functional as F

import baseline_beam_reference as BR

pytestmark = pytest.mark.gpu

# <end> made reachable but not immediate (cf. SURVEY.md 8c for the attention decoder): embedding *= emb_scale (or the
# GloVe-like fp64 table times emb_scale), linear.weight *= lin_scale, then linear.weight[END] *= end_gain and
# linear.bias[END] = end_bias.  Every case gives captions of several lengths and at least one image without a completed beam
# (asserted at k = 5 below).  lin_scale: at V = 9490 the default initialisation makes the softmax nearly flat and the top
# candidates of a step so dense that half the images meet a ranking near-tie (NEAR_TIE) within 51 steps at k = 8.
CASES = {
    "small": dict(V=131, E=24, H=32, emb_scale=30.0, lin_scale=1.0, end_gain=15.0, end_bias=-8.0, n_img=12, glove=False),
    "full": dict(V=9490, E=512, H=512, emb_scale=30.0, lin_scale=3.0, end_gain=5.0, end_bias=-6.0, n_img=16, glove=False),
    "glove": dict(V=211, E=300, H=64, emb_scale=3.0, lin_scale=1.0, end_gain=15.0, end_bias=-6.0, n_img=10, glove=True),
}
MAX_STEPS = 50
# A step whose fp64 margin (smallest gap between consecutive candidates of its top k+1, which decides the kept beams and their
# order) is below this is a near-tie that fp32-grade arithmetic does not decide: a few ulps of a running score near -100
# (one ulp = 7.6e-6).
NEAR_TIE = 2e-5


def build_decoder(case):
    import icd_b200.models.baseline as my_base
    from icd_b200 import synthetic
    p = my_base.BaselineDecoderParams()
    p.hidden_size, p.embed_size, p.vocab_size = case["H"], case["E"], case["V"]
    torch.manual_seed(0)
    dec = my_base.BaselineDecoder(p)
    V = case["V"]
    if case["glove"]:
        dec.load_pretrained_embeddins(synthetic.glove_like_table(V, case["E"]) * case["emb_scale"])
    with torch.no_grad():
        if not case["glove"]:
            dec.embedding.weight *= case["emb_scale"]
        dec.linear.weight *= case["lin_scale"]
        dec.linear.weight[V - 2] *= case["end_gain"]
        dec.linear.bias[V - 2] = case["end_bias"]
    return dec


def image_features(case, seed=5):
    return torch.randn(case["n_img"], case["E"], generator=torch.Generator().manual_seed(seed))


@functools.lru_cache(maxsize=None)
def oracle_results(name, k):
    """Per image: the fp32 and fp64 oracle outcomes (seq, ended, trace, score, per-step selection margins)."""
    case = CASES[name]
    w = {kk: v.detach().clone() for kk, v in build_decoder(case).state_dict().items()}
    w64 = {kk: v.double() for kk, v in w.items()}
    imgs = image_features(case)
    V, out = case["V"], []
    for i in range(case["n_img"]):
        r = {}
        for tag, ww, x in (("32", w, imgs[i]), ("64", w64, imgs[i].double())):
            tr, sc, mg = [], [], []
            seq, ended = BR.baseline_beam_search(ww, x, k, V - 3, V - 2, max_steps=MAX_STEPS, trace=tr, score=sc, margins=mg)
            r[tag] = (seq, ended, tr, sc, mg)
        out.append(r)
    return out


@pytest.mark.parametrize("precision", ["fp32x3", "fp32"])
@pytest.mark.parametrize("k", [1, 3, 5, 8])
@pytest.mark.parametrize("name", list(CASES))
def test_baseline_beam_matches_oracle(cuda, name, k, precision):
    from icd_b200.gen_captions import baseline_beam_search_batched
    case = CASES[name]
    V = case["V"]
    dec = build_decoder(case).to(cuda)
    imgs = image_features(case)
    with torch.no_grad():
        res = baseline_beam_search_batched(dec, imgs.to(cuda), k, V - 3, V - 2, max_steps=MAX_STEPS, want_trace=True,
                                           precision=precision)
    lens, seqs = res["len"].cpu().tolist(), res["seq"].cpu()
    scores, trace = res["score"].cpu().double(), res["trace"].cpu()
    ref = oracle_results(name, k)
    if k == 5:                                        # the recipe does what it is for
        outcomes = [len(r["64"][0]) if r["64"][1] else 0 for r in ref]
        assert 0 in outcomes and len(set(outcomes) - {0}) >= 3, outcomes
    checked = 0
    for i, r in enumerate(ref):
        seq, ended, tr, sc, mg = r["64"]
        if r["32"][:3] != r["64"][:3]:
            continue                  # the outcome is not stable under fp64 re-evaluation: not a meaningful target
        ties = [s for s, m in enumerate(mg) if m < NEAR_TIE]
        if ties:                      # the trajectory is decided up to its first near-tie selection only
            for s in range(ties[0]):
                row = trace[s, i].tolist()
                assert row[:len(tr[s])] == tr[s] and all(x == -1 for x in row[len(tr[s]):]), (i, s)
            continue
        checked += 1
        if ended:
            assert lens[i] == len(seq), (i, lens[i], seq)
            assert seqs[i, :lens[i]].tolist() == seq
            assert abs(scores[i].item() - sc[0]) <= 1e-4 * abs(sc[0]), (i, scores[i].item(), sc[0])
        else:
            assert lens[i] == 0
        for s, words in enumerate(tr):
            row = trace[s, i].tolist()
            assert row[:len(words)] == words and all(x == -1 for x in row[len(words):]), (i, s)
        assert bool((trace[len(tr):, i] == -1).all()), i
    assert 2 * checked >= len(ref), "only %d of %d images are stable under fp64" % (checked, len(ref))


def _mixed_features(case):
    base = image_features(case)
    g = torch.Generator().manual_seed(11)
    return torch.cat([base, base.flip(0) * 0.7 + 0.1, torch.randn(base.shape, generator=g) * 1.5], dim=0)


@pytest.mark.parametrize("precision", ["fp32", "fp32x3"])
def test_baseline_beam_batch_equals_single_images_and_chunks(cuda, precision):
    """Finished beams and images leave the working set (device-side compaction): an image's result must not depend on
    which images share the call, nor on how the images are chunked."""
    from icd_b200.gen_captions import baseline_beam_search_batched
    case = CASES["small"]
    V, k = case["V"], 4
    dec = build_decoder(case).to(cuda)
    feats = _mixed_features(case).to(cuda)
    with torch.no_grad():
        full = baseline_beam_search_batched(dec, feats, k, V - 3, V - 2, max_steps=30, want_trace=True, precision=precision)
        lens = full["len"].cpu().tolist()
        assert len(set(lens)) >= 3 and 0 in lens, "the test needs images that finish at different steps"
        for i in range(feats.shape[0]):
            one = baseline_beam_search_batched(dec, feats[i:i + 1], k, V - 3, V - 2, max_steps=30, want_trace=True,
                                               precision=precision)
            assert torch.equal(one["len"][0], full["len"][i])
            assert torch.equal(one["seq"][0], full["seq"][i])
            assert torch.equal(one["score"][0], full["score"][i])
            assert torch.equal(one["trace"][:, 0], full["trace"][:, i])
        chunked = baseline_beam_search_batched(dec, feats, k, V - 3, V - 2, max_steps=30, want_trace=True, chunk=2,
                                               precision=precision)
    for key in ("len", "seq", "score", "trace"):
        assert torch.equal(chunked[key], full[key]), key


def test_baseline_beam_is_deterministic(cuda):
    from icd_b200.gen_captions import baseline_beam_search_batched
    case = CASES["full"]
    V = case["V"]
    dec = build_decoder(case).to(cuda)
    feats = image_features(case).to(cuda)
    with torch.no_grad():
        a = baseline_beam_search_batched(dec, feats, 5, V - 3, V - 2, want_trace=True)
        b = baseline_beam_search_batched(dec, feats, 5, V - 3, V - 2, want_trace=True)
    for key in ("len", "seq", "score", "trace"):
        assert torch.equal(a[key], b[key]), key


@pytest.mark.parametrize("name", ["full", "glove"])
def test_baseline_beam_agrees_with_the_training_forward(cuda, name):
    """Greedy captions are the argmax of the teacher-forced forward fed with themselves (wherever the top-2 margin is not a
    near-tie), and a k = 5 winner's score is the teacher-forced log-probability of its caption over positions t >= 1."""
    from icd_b200.gen_captions import baseline_beam_search_batched
    case = dict(CASES[name], end_bias=CASES[name]["end_bias"] + 2.0)      # more greedy captions complete
    V = case["V"]
    dec = build_decoder(case).to(cuda)
    feats = image_features(case).to(cuda)
    checked_greedy = checked_score = 0
    with torch.no_grad():
        g = baseline_beam_search_batched(dec, feats, 1, V - 3, V - 2)
        b = baseline_beam_search_batched(dec, feats, 5, V - 3, V - 2)
        for i in range(case["n_img"]):
            L = int(g["len"][i])
            if L:
                cap = g["seq"][i:i + 1, :L].long()
                out = dec(feats[i:i + 1], cap)[0]                               # fp32 tier forward, (L, V)
                top2 = out.topk(2, dim=1).values
                for t in range(1, L):
                    if float(top2[t, 0] - top2[t, 1]) > 1e-4:
                        assert int(out[t].argmax()) == int(cap[0, t]), (i, t)
                checked_greedy += 1
            L = int(b["len"][i])
            if L:
                cap = b["seq"][i:i + 1, :L].long()
                lp = F.log_softmax(dec(feats[i:i + 1], cap)[0].double(), dim=1)
                tf = float(sum(lp[t, int(cap[0, t])] for t in range(1, L)))
                got = float(b["score"][i])
                assert abs(got - tf) <= 1e-4 * abs(tf), (i, got, tf)
                checked_score += 1
    assert checked_greedy >= 1 and checked_score >= 1


def test_baseline_caption_image_drop_in(cuda, capsys):
    from icd_b200.gen_captions import (baseline_beam_search_batched, baseline_caption_image_beam_search,
                                       beam_search_sharded)
    from icd_b200.vocabulary import synthetic_vocab
    case = CASES["small"]
    V = case["V"]
    vocab = synthetic_vocab(V)
    dec = build_decoder(case).to(cuda)
    feats = image_features(case).to(cuda)

    class Args:
        beam_size = 5

    class Identity(torch.nn.Module):
        def forward(self, x):
            return x

    with torch.no_grad():
        res = baseline_beam_search_batched(dec, feats, 5, V - 3, V - 2, want_trace=True)
    i = [j for j in range(case["n_img"]) if int(res["len"][j]) > 0][0]
    capsys.readouterr()
    seq, ended = baseline_caption_image_beam_search(cuda, Args, feats[i:i + 1], Identity(), dec, vocab)
    printed = [ln for ln in capsys.readouterr().out.strip().split("\n") if ln]
    assert ended is True and seq == res["seq"][i, :int(res["len"][i])].tolist()
    assert seq[0] == vocab("<start>") and seq[-1] == vocab("<end>")
    rows = [[x for x in row if x >= 0] for row in res["trace"][:, i].tolist()]
    assert printed == [str([vocab.i2w[x] for x in row]) for row in rows if row]

    with torch.no_grad():                                                  # <end> suppressed: the failure tuple
        dec.linear.bias[V - 2] = -1e4
    assert baseline_caption_image_beam_search(cuda, Args, feats[i:i + 1], Identity(), dec, vocab) == \
        ([V - 3, V - 2], False)
    with torch.no_grad():
        dec.linear.bias[V - 2] = case["end_bias"]

    with pytest.raises(ValueError):
        baseline_beam_search_batched(dec, feats, 5, V - 3, V - 2, precision="bf16")

    with torch.no_grad():
        sh = beam_search_sharded(dec, feats, 5, V - 3, V - 2)
    for key in ("len", "seq", "score"):
        assert torch.equal(sh[key], res[key]), key
