"""CPU tier: the beam search over the BaselineDecoder (tests/baseline_beam_reference.py) and its C ABI argument checks.

The reference has no generation function for the baseline decoder; baseline_beam_reference.py defines one (the attention
beam search's state machine over the baseline step, with the image feature as an unscored step 0).  These tests tie that
definition to things the reference does have: the pinned oracle of the attention beam search, the module's own nn.LSTM /
nn.Linear stepped greedily, and the teacher-forced forward."""
import ctypes

import pytest
import torch
import torch.nn.functional as F

from oracle import decoders as O

import baseline_beam_reference as BR
import helpers as Hh

SMALL = dict(V=131, E=24, H=32, emb_scale=30.0, end_gain=15.0, end_bias=-8.0)


def baseline_module(case, wseed=0):
    import icd_b200.models.baseline as my_base
    p = my_base.BaselineDecoderParams()
    p.hidden_size, p.embed_size, p.vocab_size = case["H"], case["E"], case["V"]
    torch.manual_seed(wseed)
    dec = my_base.BaselineDecoder(p)
    V = case["V"]
    with torch.no_grad():                                    # <end> reachable but not immediate: captions of varied length
        dec.embedding.weight *= case["emb_scale"]
        dec.linear.weight[V - 2] *= case["end_gain"]
        dec.linear.bias[V - 2] = case["end_bias"]
    return dec


def images(n, E, seed=5):
    return torch.randn(n, E, generator=torch.Generator().manual_seed(seed))


def greedy_rollout(dec, img, start_id, end_id, max_steps):
    """Step the module's own nn.LSTM / nn.Linear one token at a time (CPU), argmax at every step."""
    with torch.no_grad():
        _, state = dec.lstm(img.view(1, 1, -1))                                  # step 0: the image feature, not scored
        seq, prev = [start_id], start_id
        for _ in range(max_steps + 1):
            x = dec.embedding(torch.tensor([[prev]])).to(img.dtype)
            out, state = dec.lstm(x, state)
            prev = int(dec.linear(out[:, 0]).argmax(dim=1))
            seq.append(prev)
            if prev == end_id:
                return seq, True
    return [start_id, end_id], False


@pytest.mark.parametrize("k", [1, 3, 8])
def test_state_machine_with_the_attention_step_equals_the_oracle_beam_search(k):
    """The state machine the baseline search is built on is the reference's: run with the attention decoder's step it gives
    oracle.decoders.beam_search's captions, outcomes and per-step candidate words (that oracle is pinned to the unmodified
    reference by the golden tests)."""
    import icd_b200.models.attention as my_att
    from icd_b200.vocabulary import synthetic_vocab
    case = dict(Hh.BEAM_CASES["beam_small"], dropout=0.5, train=False, fine_tune_embedding=True)
    dec = Hh.build_attention_module(case, my_att.AttentionDecoder, my_att.AttentionDecoderParams, synthetic_vocab(case["V"]))
    Hh.apply_beam_recipe(dec, case)
    w = {kk: v.detach().double() for kk, v in dec.state_dict().items()}
    feats = Hh.beam_features(case).double()
    V = case["V"]
    outcomes = set()
    for i in range(feats.shape[0]):
        tr_o, tr_m = [], []
        seq, _, ended = O.beam_search(w, feats[i:i + 1], k, V - 3, V - 2, trace=tr_o)
        step, enc = BR.attention_step(w, feats[i:i + 1])
        h, c = O.init_hidden_state(w, enc)
        P, C = enc.shape[1], enc.shape[2]
        got = BR.beam_state_machine(step, (enc.expand(k, P, C), h.expand(k, -1), c.expand(k, -1)), k, V, torch.float64,
                                    V - 3, V - 2, trace=tr_m)
        assert got == (seq, ended) and tr_m == tr_o, (k, i)
        outcomes.add(len(seq) if ended else 0)
    assert len(outcomes) >= 2


def test_greedy_beam_equals_stepping_the_modules_lstm():
    """beam_size 1 is greedy decoding: the oracle equals an argmax rollout of the module's own nn.LSTM / nn.Linear."""
    V = SMALL["V"]
    outcomes = set()
    for end_bias in (-8.0, -3.0):
        case = dict(SMALL, end_bias=end_bias)
        dec = baseline_module(case).double()
        w = {k: v.detach().clone() for k, v in dec.state_dict().items()}
        imgs = images(12, case["E"]).double()
        for i in range(imgs.shape[0]):
            for max_steps in (50, 5):
                ref = greedy_rollout(dec, imgs[i], V - 3, V - 2, max_steps)
                got = BR.baseline_beam_search(w, imgs[i], 1, V - 3, V - 2, max_steps=max_steps)
                assert got == ref, (end_bias, i, max_steps)
                outcomes.add(len(got[0]) if got[1] else 0)
    assert 0 in outcomes and len(outcomes) >= 3        # failures and completed captions of several lengths


@pytest.mark.parametrize("k", [3, 5])
def test_winner_score_is_the_teacher_forced_log_prob_of_its_caption(k):
    """Scored steps are t >= 1 of the training forward fed with the caption itself: score = sum_t log_softmax(out)[t, seq[t]]."""
    case = SMALL
    V = case["V"]
    w = {kk: v.detach().double() for kk, v in baseline_module(case).state_dict().items()}
    imgs = images(12, case["E"]).double()
    lengths = set()
    for i in range(imgs.shape[0]):
        score = []
        seq, ended = BR.baseline_beam_search(w, imgs[i], k, V - 3, V - 2, score=score)
        if not ended:
            assert seq == [V - 3, V - 2] and score == []
            continue
        assert seq[0] == V - 3 and seq[-1] == V - 2 and (V - 2) not in seq[1:-1]
        lengths.add(len(seq))
        cap = torch.tensor([seq])
        lp = F.log_softmax(O.baseline_decoder_forward(w, imgs[i:i + 1], cap), dim=2)[0]
        tf = float(sum(lp[t, seq[t]] for t in range(1, len(seq))))
        assert abs(score[0] - tf) <= 1e-9 * abs(tf), (i, score[0], tf)
    assert len(lengths) >= 3


def test_fp64_glove_table_equals_its_fp32_cast():
    from icd_b200 import synthetic
    V, E, H = 211, 300, 64
    case = dict(V=V, E=E, H=H, emb_scale=1.0, end_gain=15.0, end_bias=-6.0)
    w = {k: v.detach().clone() for k, v in baseline_module(case, wseed=3).state_dict().items()}
    w64 = dict(w, **{"embedding.weight": synthetic.glove_like_table(V, E) * 3.0})
    assert w64["embedding.weight"].dtype == torch.float64
    w32 = dict(w, **{"embedding.weight": w64["embedding.weight"].float()})
    imgs = images(8, E)
    for i in range(imgs.shape[0]):
        t64, t32 = [], []
        s64, s32 = [], []
        assert (BR.baseline_beam_search(w64, imgs[i], 5, V - 3, V - 2, trace=t64, score=s64) ==
                BR.baseline_beam_search(w32, imgs[i], 5, V - 3, V - 2, trace=t32, score=s32))
        assert t64 == t32 and s64 == s32


# ------------------------------------------------------------------------------------------------------------ C ABI
def _desc(**over):
    from icd_b200 import _lib
    d = _lib.BaseBeamDesc()
    fake = 256                                   # never dereferenced: the arguments are refused before any CUDA call
    kw = dict(n_img=4, k=5, max_steps=50, E=512, H=512, V=9490, precision=_lib.PREC_FP32X3, emb_is_f64=0,
              start_id=9487, end_id=9488, img_features=fake, emb_w=fake, w_ih=fake, w_hh=fake, b_ih=fake, b_hh=fake,
              lin_w=fake, lin_b=fake, out_len=fake, out_seq=fake, out_score=fake, ws=fake)
    kw.update(over)
    for k, v in kw.items():
        setattr(d, k, v)
    return d


def test_base_beam_desc_layout_matches_the_library():
    from icd_b200 import _lib
    L = _lib.lib()
    assert L.icd_sizeof_base_beam_desc() == ctypes.sizeof(_lib.BaseBeamDesc)
    for name in ("icd_baseline_beam_search", "icd_baseline_beam_search_ws_bytes", "icd_sizeof_base_beam_desc"):
        assert hasattr(L, name)
    d = _desc()
    need = L.icd_baseline_beam_search_ws_bytes(ctypes.byref(d))
    d2 = _desc(precision=_lib.PREC_FP32)
    assert need > L.icd_baseline_beam_search_ws_bytes(ctypes.byref(d2)) > 0       # the fp32x3 tier adds the weight splits


@pytest.mark.parametrize("what,over,msg", [
    ("k=9", dict(k=9), b"k in 1..8"),
    ("k=0", dict(k=0), b"k in 1..8"),
    ("bf16", dict(precision=1), b"precision"),
    ("too many rows", dict(n_img=20000, k=4), b"65535"),
    ("E not a multiple of 4", dict(E=302), b"multiples of 4"),
    ("V < k", dict(V=4, start_id=1, end_id=2), b"smaller than the beam"),
    ("small workspace", dict(), b"workspace too small"),
])
def test_argument_errors_are_refused_without_a_gpu(what, over, msg):
    from icd_b200 import _lib
    L = _lib.lib()
    d = _desc(**over)
    need = L.icd_baseline_beam_search_ws_bytes(ctypes.byref(d))
    if what == "small workspace":
        d.ws_bytes = need - 1
    else:
        assert need == -1 and msg in L.icd_last_error_string(), what      # the size query refuses the shape too
        d.ws_bytes = 1 << 40
    rc = L.icd_baseline_beam_search(ctypes.byref(d), None)
    assert rc < 0, what
    assert msg in L.icd_last_error_string(), (what, L.icd_last_error_string())
