"""GPU tier: seeded caption sampling (gen_captions.sample_captions; icd_sample_captions, icd_baseline_sample_captions)
against its definition (tests/sampling_reference.py), against the beam search's greedy limit, against itself (batching,
chunking, sample groups, seeds) and against the training forward of the same module."""
import functools

import numpy as np
import pytest
import torch
import torch.nn.functional as F
from scipy import stats

import helpers as Hh
import sampling_reference as SR
from test_gpu_baseline_beam import CASES as BASE_CASES, build_decoder, image_features

pytestmark = pytest.mark.gpu

MAX_STEPS = 30
# A step whose fp64 decision margin (gap between the two largest keys, at the top-k boundary, or the top-2 logit gap for greedy)
# is below this is a near-tie the fp32-grade logits do not decide: the tier's logit error is ~1e-5 relative on logits of a
# few units after up to 31 recurrent steps, and a key adds l / T (T >= 0.7) and an fp32 Gumbel term (~2 ulps of ~10).
NEAR_TIE = 2e-4
COMBOS = [(1, 0.0, 0), (5, 0.7, 10), (8, 1.0, 0), (5, 1.5, 1), (8, 1.0, 10)]      # (m, temperature, top_k)
SEED = 0x5EED5EED1234


def _att_setup(end_bias=None):
    import icd_b200.models.attention as my_att
    from icd_b200.vocabulary import synthetic_vocab
    case = dict(Hh.BEAM_CASES["beam_small"], dropout=0.5, train=False, fine_tune_embedding=True)
    if end_bias is not None:
        case["end_bias"] = end_bias
    dec = Hh.build_attention_module(case, my_att.AttentionDecoder, my_att.AttentionDecoderParams, synthetic_vocab(case["V"]))
    Hh.apply_beam_recipe(dec, case)
    return dec, Hh.beam_features(case), case["V"]


def make_case(name):
    """-> (module on CPU, features on CPU, V, reference start function).  "full_ending": the full size with <end> made more
    likely (as the beam tests' training-forward check does), so that greedy captions complete within MAX_STEPS.  "att_ending":
    the attention case with fc.bias[<end>] = +2, where samples at T = 1 end anywhere from step 2 to past the cap (at -2 none
    ends within 31 steps), so that compaction is exercised."""
    if name in ("att_small", "att_ending"):
        dec, feats, V = _att_setup(2.0 if name == "att_ending" else None)
        return dec, feats, V, SR.attention_start
    if name == "full_ending":
        case = dict(BASE_CASES["full"], end_bias=BASE_CASES["full"]["end_bias"] + 2.0)
        return build_decoder(case), image_features(case), case["V"], SR.baseline_start
    case = dict(BASE_CASES[name])
    if name == "full":
        case["n_img"] = 3
    return build_decoder(case), image_features(case), case["V"], SR.baseline_start


@functools.lru_cache(maxsize=None)
def reference(name, m, temperature, top_k):
    dec, feats, V, start = make_case(name)
    w = {k: v.detach().double() for k, v in dec.state_dict().items()}
    out = []
    for i in range(feats.shape[0]):
        step, st = start(w, feats[i:i + 1].double() if name == "att_small" else feats[i].double())
        out.append(SR.sample_image(step, st, m, V - 3, V - 2, MAX_STEPS, temperature, top_k, SEED, i))
    return out


def run(dec, feats, cuda, V, m, temperature, top_k, precision="fp32x3", **kw):
    from icd_b200.gen_captions import sample_captions
    with torch.no_grad():
        return sample_captions(dec.to(cuda), feats.to(cuda), m, V - 3, V - 2, temperature=temperature, top_k=top_k,
                               seed=SEED, max_steps=MAX_STEPS, want_logp=True, precision=precision, **kw)


@pytest.mark.parametrize("precision", ["fp32x3", "fp32"])
@pytest.mark.parametrize("combo", range(len(COMBOS)))
@pytest.mark.parametrize("name", ["small", "full", "glove", "att_small"])
def test_samples_match_the_reference(cuda, name, combo, precision):
    m, T, top_k = COMBOS[combo]
    if name == "full" and m == 8:
        pytest.skip("the fp64 reference of 8 samples at V = 9490 is slow on the CPU; m = 1 and 5 cover the full size")
    dec, feats, V, _ = make_case(name)
    res = run(dec, feats, cuda, V, m, T, top_k, precision)
    seq, ln, ended = res["seq"].cpu(), res["len"].cpu(), res["ended"].cpu()
    score, logp = res["score"].cpu().double(), res["logp"].cpu().double()
    ref = reference(name, m, T, top_k)
    checked = total = 0
    for i, samples in enumerate(ref):
        for j, r in enumerate(samples):
            total += 1
            ties = [s for s, mg in enumerate(r["margins"]) if mg < NEAR_TIE]
            upto = ties[0] if ties else len(r["margins"])          # steps decided before the first near-tie
            got = seq[i, j].tolist()
            assert got[:upto + 1] == r["seq"][:upto + 1], (i, j, upto)
            assert np.allclose(logp[i, j, :upto].numpy(), r["logp"][:upto], atol=1e-4, rtol=0), (i, j)
            if ties:
                continue
            checked += 1
            assert int(ln[i, j]) == r["len"] and bool(ended[i, j]) == r["ended"], (i, j)
            assert got[r["len"]:] == [0] * (MAX_STEPS + 2 - r["len"]), (i, j)
            assert bool((logp[i, j, r["len"] - 1:] == 0).all()), (i, j)
            assert abs(score[i, j].item() - r["score"]) <= 1e-4 * max(1.0, abs(r["score"])), (i, j, score[i, j].item(), r["score"])
    assert 2 * checked >= total, "only %d of %d samples are free of near-ties" % (checked, total)


@pytest.mark.parametrize("precision", ["fp32x3", "fp32"])
@pytest.mark.parametrize("name", ["full_ending", "att_small"])
def test_greedy_sampling_is_the_k1_beam_search(cuda, name, precision):
    from icd_b200.gen_captions import baseline_beam_search_batched, beam_search_batched
    dec, feats, V, _ = make_case(name)
    dec = dec.to(cuda)
    x = feats.to(cuda)
    beam = baseline_beam_search_batched if name != "att_small" else functools.partial(beam_search_batched, want_alphas=False)
    with torch.no_grad():
        b = beam(dec, x, 1, V - 3, V - 2, max_steps=MAX_STEPS, want_trace=True, precision=precision)
    s = run(dec, feats, cuda, V, 1, 0.0, 0, precision)
    ended_any = 0
    for i in range(feats.shape[0]):
        L = int(b["len"][i])
        if L:
            ended_any += 1
            assert int(s["len"][i, 0]) == L and int(s["ended"][i, 0]) == 1
            assert torch.equal(s["seq"][i, 0, :L], b["seq"][i, :L])
            assert abs(float(s["score"][i, 0]) - float(b["score"][i])) <= 1e-6 * abs(float(b["score"][i]))
        else:
            assert int(s["ended"][i, 0]) == 0
            assert s["seq"][i, 0, 1:].tolist() == b["trace"][:, i, 0].tolist()
    assert ended_any >= 1


@pytest.mark.parametrize("precision", ["fp32x3", "fp32"])
@pytest.mark.parametrize("name", ["small", "att_ending"])
def test_sampling_does_not_depend_on_batching_chunking_or_groups(cuda, name, precision):
    dec, feats, V, _ = make_case(name)
    keys = ("seq", "len", "ended", "score", "logp")
    full = run(dec, feats, cuda, V, 5, 1.0, 10, precision)
    assert len(set(full["len"].flatten().tolist())) >= 2 and 0 < int(full["ended"].sum()) < full["ended"].numel(), \
        "the test needs samples that end at different steps and samples that are truncated"
    per_image = run(dec, feats, cuda, V, 5, 1.0, 10, precision, chunk=1)      # one call per image, img_base = its index
    for k in keys:
        assert torch.equal(per_image[k], full[k]), k
    chunked = run(dec, feats, cuda, V, 5, 1.0, 10, precision, chunk=2)
    for k in keys:
        assert torch.equal(chunked[k], full[k]), k
    twelve = run(dec, feats, cuda, V, 12, 1.0, 10, precision)
    first = run(dec, feats, cuda, V, 8, 1.0, 10, precision)
    rest = run(dec, feats, cuda, V, 4, 1.0, 10, precision, sample_base=8)
    for k in keys:
        assert torch.equal(twelve[k], torch.cat([first[k], rest[k]], dim=1)), k
        assert torch.equal(twelve[k][:, :5], full[k]), k
    allk = run(dec, feats, cuda, V, 5, 1.0, V, precision)
    nok = run(dec, feats, cuda, V, 5, 1.0, 0, precision)
    for k in keys:
        assert torch.equal(allk[k], nok[k]), k


def test_seeds_and_image_indices(cuda):
    from icd_b200.gen_captions import sample_captions
    dec, feats, V, _ = make_case("small")
    dec = dec.to(cuda)
    same = feats[:1].repeat(6, 1).to(cuda)
    with torch.no_grad():
        a = sample_captions(dec, same, 4, V - 3, V - 2, seed=11, max_steps=MAX_STEPS)
        b = sample_captions(dec, same, 4, V - 3, V - 2, seed=11, max_steps=MAX_STEPS)
        c = sample_captions(dec, same, 4, V - 3, V - 2, seed=12, max_steps=MAX_STEPS)
        torch.manual_seed(99)
        d1 = sample_captions(dec, same, 4, V - 3, V - 2, max_steps=MAX_STEPS)
        torch.manual_seed(99)
        d2 = sample_captions(dec, same, 4, V - 3, V - 2, max_steps=MAX_STEPS)
    for k in ("seq", "len", "ended", "score"):
        assert torch.equal(a[k], b[k]), k
        assert torch.equal(d1[k], d2[k]), k
    assert a["seed"] == 11 and d1["seed"] == d2["seed"]
    assert not torch.equal(a["seq"], c["seq"])
    flat = [tuple(r) for r in a["seq"].reshape(-1, MAX_STEPS + 2).tolist()]
    assert len(set(flat)) > len(flat) // 2, "identical images at different indices must draw different samples"


@pytest.mark.parametrize("name", ["full", "glove"])
def test_logp_is_the_teacher_forced_log_softmax(cuda, name):
    dec, feats, V, _ = make_case(name)
    dec = dec.to(cuda)
    x = feats.to(cuda)
    res = run(dec, feats, cuda, V, 4, 1.0, 0, "fp32x3")
    n = 0
    with torch.no_grad():
        for i in range(x.shape[0]):
            for j in range(4):
                L = int(res["len"][i, j])
                cap = res["seq"][i, j:j + 1, :L].long()
                lp = F.log_softmax(dec(x[i:i + 1], cap)[0].double(), dim=1)
                tf = torch.stack([lp[t, int(cap[0, t])] for t in range(1, L)])
                assert torch.allclose(res["logp"][i, j, :L - 1].double(), tf, atol=1e-4, rtol=0), (i, j)
                assert abs(float(res["score"][i, j]) - float(tf.sum())) <= 1e-4 * max(1.0, abs(float(tf.sum()))), (i, j)
                n += 1
    assert n == 4 * x.shape[0]


@pytest.mark.parametrize("temperature,top_k", [(1.0, 10), (0.7, 0)])
def test_first_step_distribution(cuda, temperature, top_k):
    """4096 identical images x 8 samples at a fixed seed: step-1 tokens against the fp64 softmax(l / T) over the top-k."""
    from icd_b200.gen_captions import sample_captions
    dec, feats, V, _ = make_case("small")
    w = {k: v.detach().double() for k, v in dec.state_dict().items()}
    step, st = SR.baseline_start(w, feats[0].double())
    l = step(st, torch.tensor([[V - 3]]))[0][0]
    cand = SR.candidates(l.numpy(), top_k)
    p = torch.softmax(l[torch.as_tensor(cand)] / temperature, dim=0).numpy()
    with torch.no_grad():
        res = sample_captions(dec.to(cuda), feats[:1].repeat(4096, 1).to(cuda), 8, V - 3, V - 2, temperature=temperature,
                              top_k=top_k, seed=2024, max_steps=1)
    tok = res["seq"][:, :, 1].reshape(-1).cpu().numpy()
    counts = np.bincount(tok, minlength=V)
    s = np.sort(l.numpy())[::-1]
    if top_k and s[top_k - 1] - s[top_k] > NEAR_TIE:
        assert counts[np.setdiff1d(np.arange(V), cand)].sum() == 0
    obs, exp = counts[cand], p * tok.size
    big = exp >= 5
    obs = np.append(obs[big], obs[~big].sum())
    exp = np.append(exp[big], exp[~big].sum())
    if exp[-1] == 0:
        obs, exp = obs[:-1], exp[:-1]
    assert stats.chisquare(obs, exp * obs.sum() / exp.sum()).pvalue > 1e-3


def test_refusals(cuda):
    from icd_b200 import _lib
    from icd_b200.gen_captions import sample_captions
    dec, feats, V, _ = make_case("small")
    dec = dec.to(cuda)
    x = feats.to(cuda)
    with pytest.raises(ValueError):
        sample_captions(dec, x, 2, V - 3, V - 2, precision="bf16")
    with pytest.raises(ValueError):
        sample_captions(dec, x, 0, V - 3, V - 2)
    with pytest.raises(_lib.IcdError):
        sample_captions(dec, x, 2, V - 3, V - 2, top_k=V + 1)
    with pytest.raises(_lib.IcdError):
        sample_captions(dec, x, 2, V - 3, V - 2, temperature=-1.0)
    with pytest.raises(_lib.IcdError):
        sample_captions(dec, x, 2, V - 3, V - 2, temperature=float("nan"))
