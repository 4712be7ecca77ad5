"""TEST INFRASTRUCTURE ONLY: beam search over the BaselineDecoder, restated on the CPU (torch, dtype-generic).

The reference has no generation function for the baseline decoder, so this module defines the semantics
``icd_baseline_beam_search`` implements: the beam state machine of gen_captions.py:44-127 (``oracle.decoders.beam_search``,
SURVEY.md Appendix C) with the decoder step abstracted, and the BaselineDecoder's step plugged into it.
``tests/test_baseline_beam_oracle.py`` pins ``beam_state_machine`` to ``oracle.decoders.beam_search`` (the attention step
run through it gives the oracle's captions and traces) and ``baseline_beam_search`` to the module's own nn.LSTM and to the
teacher-forced forward.
"""
import torch
import torch.nn.functional as F

from oracle.decoders import init_hidden_state, lstm_cell, soft_attention


def beam_state_machine(step_fn, state, k, V, dtype, start_id, end_id, max_steps=50, trace=None, score=None, margins=None):
    """The beam loop of gen_captions.py:44-127 for one image, with the decoder step abstracted.

    ``state``: tuple of per-beam tensors (first dim k) that follow the beams (h, c, ...).
    ``step_fn(state, k_prev_words (k, 1)) -> (logits (k, V), state)``: one decoder step.
    Returns (seq, caption_end) of the winner, ([start, end], False) when no beam completed.  ``trace`` (list) receives the
    next-word ids per step (:91), ``score`` (list) the winner's raw summed log-prob, ``margins`` (list) per step the smallest
    gap between consecutive candidates of the step's top k+1 — the ranking that decides which candidates are kept and in
    which beam order — which tells a test where a selection is a near-tie."""
    k_prev_words = torch.full((k, 1), start_id, dtype=torch.long)             # :47
    seqs = torch.full((k, 1), start_id, dtype=torch.long)                     # :50
    top_k_scores = torch.zeros(k, 1, dtype=dtype)                              # :52
    complete_seqs, complete_scores = [], []
    caption_end = False
    step = 1
    while True:
        logits, state = step_fn(state, k_prev_words)                          # :65-72
        scores = F.log_softmax(logits, dim=1)                                  # :74
        scores = top_k_scores.expand_as(scores) + scores                       # :76
        cand = scores[0] if step == 1 else scores.view(-1)                     # :78-82
        top_k_scores, top_k_words = cand.topk(k, 0, True, True)
        if margins is not None:
            top = cand.topk(min(k + 1, cand.numel()))[0]
            margins.append(float((top[:-1] - top[1:]).min()) if top.numel() > 1 else float("inf"))
        prev_word_inds = top_k_words // V                                      # :85
        next_word_inds = top_k_words % V                                       # :86
        seqs = torch.cat([seqs[prev_word_inds], next_word_inds.unsqueeze(1)], dim=1)         # :88
        if trace is not None:
            trace.append(next_word_inds.tolist())                              # :91 (print)
        incomplete = [i for i, nw in enumerate(next_word_inds.tolist()) if nw != end_id]     # :93-94
        complete = sorted(set(range(len(next_word_inds))) - set(incomplete))   # :96
        if len(complete) > 0:                                                  # :99-103
            caption_end = True
            complete_seqs.extend(seqs[complete].tolist())
            complete_scores.extend(top_k_scores[complete])
        k -= len(complete)                                                     # :104
        if k == 0:                                                             # :107
            break
        seqs = seqs[incomplete]                                                # :109-116
        state = tuple(t[prev_word_inds[incomplete]] for t in state)
        top_k_scores = top_k_scores[incomplete].unsqueeze(1)
        k_prev_words = next_word_inds[incomplete].unsqueeze(1)
        if step > max_steps:                                                   # :119
            break
        step += 1
    if not caption_end:                                                        # :123-125
        return [start_id, end_id], False
    idx = complete_scores.index(max(complete_scores))                          # :127 first max
    if score is not None:
        score.append(float(complete_scores[idx]))
    return complete_seqs[idx], True


def attention_step(w, encoder_out):
    """(step_fn, initial state) of the attention decoder (gen_captions.py:41-72, as oracle.decoders.beam_search), for the
    test that pins ``beam_state_machine`` to the oracle."""
    dtype = w["fc.weight"].dtype
    C = encoder_out.size(-1)
    enc = encoder_out.reshape(1, -1, C).to(dtype)

    def step(state, k_prev_words):
        enc, h, c = state
        emb = F.embedding(k_prev_words, w["embedding.weight"]).squeeze(1)
        awe, _ = soft_attention(w, enc, h)
        awe = torch.sigmoid(F.linear(h, w["f_beta.weight"], w["f_beta.bias"])) * awe
        x = torch.cat([emb.double(), awe.double()], dim=1).to(dtype)
        h, c = lstm_cell(x, h, c, w["decode_step.weight_ih"], w["decode_step.weight_hh"],
                         w["decode_step.bias_ih"], w["decode_step.bias_hh"])
        return F.linear(h, w["fc.weight"], w["fc.bias"]), (enc, h, c)

    return step, enc


def baseline_beam_search(w, img_features, beam_size, start_id, end_id, max_steps=50, trace=None, score=None, margins=None):
    """Beam search over the BaselineDecoder (models/baseline.py:81-111 run autoregressively), one image:
    ``img_features`` (E,) or (1, E), what the baseline encoder returns.  Returns (seq, Caption_End); on failure
    ([start, end], False).

    Step 0: x_0 = the image feature, cast to the weights' dtype (:101), one LSTM step from the zero state (:106); its
    logits are NOT scored and position 0 of every caption is <start> — teacher forcing trains outputs[:, 0] against
    captions[:, 0] = <start> (:93-109), so the first real prediction is conditioned on emb(<start>).  Steps 1 ..
    max_steps+1 are ``beam_state_machine`` with the baseline step: emb(previous word) cast to the weights' dtype (an fp64
    GloVe table included, :101), one LSTM step, log_softmax(linear(h)) plus the running score.  The winner is the first
    completed beam with the maximal raw summed log-prob.  beam_size 1 is greedy decoding.  ``trace``, ``score``, ``margins``
    as in ``beam_state_machine``."""
    dtype = w["linear.weight"].dtype
    k = beam_size
    V = w["linear.weight"].size(0)
    H = w["lstm.weight_hh_l0"].size(1)
    cell = (w["lstm.weight_ih_l0"], w["lstm.weight_hh_l0"], w["lstm.bias_ih_l0"], w["lstm.bias_hh_l0"])
    x0 = img_features.reshape(1, -1).to(dtype)                                 # :101 (.float() there)
    zero = torch.zeros(1, H, dtype=dtype)
    h0, c0 = lstm_cell(x0, zero, zero, *cell)                                  # step 0 from the zero state (:106)

    def step(state, k_prev_words):
        h, c = state
        x = F.embedding(k_prev_words, w["embedding.weight"]).squeeze(1).to(dtype)   # :97, :101
        h, c = lstm_cell(x, h, c, *cell)
        return F.linear(h, w["linear.weight"], w["linear.bias"]), (h, c)          # :109

    return beam_state_machine(step, (h0.expand(k, H), c0.expand(k, H)), k, V, dtype, start_id, end_id, max_steps,
                              trace, score, margins)
