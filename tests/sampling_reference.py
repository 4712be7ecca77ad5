"""TEST INFRASTRUCTURE ONLY: seeded caption sampling restated on the CPU (numpy / torch, dtype-generic).

This module states what ``icd_sample_captions`` / ``icd_baseline_sample_captions`` compute (include/icd_b200.h):
- ``philox4x32_10``: the counter-based generator, vectorised over counters;
- ``gumbel``: u = ((bits >> 8) + 0.5) * 2^-24 and g = -log(-log(u)), in fp64;
- ``select``: one step's draw (greedy, or Gumbel-max over the top-k candidates) with its decision margins;
- ``sample_image``: the per-sample loop over an abstract decoder step, from the start state the beam searches use.
The decoder steps are those of ``baseline_beam_reference`` (the baseline step from ``oracle.decoders.lstm_cell``, and
``attention_step``), so a sample's start state is exactly the beam search's.
"""
import numpy as np
import torch
import torch.nn.functional as F

import baseline_beam_reference as BR
from oracle.decoders import init_hidden_state, lstm_cell

_M0, _M1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
_W0, _W1 = 0x9E3779B9, 0xBB67AE85
_MASK = np.uint64(0xFFFFFFFF)


def philox4x32_10(c0, c1, c2, c3, k0, k1):
    """Philox4x32-10 (Salmon et al. 2011) over arrays of counters (broadcast), key (k0, k1) -> four uint32 arrays."""
    c = [np.asarray(x, dtype=np.uint64) & _MASK for x in np.broadcast_arrays(c0, c1, c2, c3)]
    k0, k1 = int(k0) & 0xFFFFFFFF, int(k1) & 0xFFFFFFFF
    for _ in range(10):
        p0, p1 = _M0 * c[0], _M1 * c[2]
        hi0, lo0 = p0 >> np.uint64(32), p0 & _MASK
        hi1, lo1 = p1 >> np.uint64(32), p1 & _MASK
        c = [hi1 ^ c[1] ^ np.uint64(k0), lo1, hi0 ^ c[3] ^ np.uint64(k1), lo0]
        k0, k1 = (k0 + _W0) & 0xFFFFFFFF, (k1 + _W1) & 0xFFFFFFFF
    return [x.astype(np.uint32) for x in c]


def token_bits(seed, step, img, sample, V):
    """(V,) uint32: word v % 4 of Philox(counter = (v / 4, step, img, sample), key = (seed lo, seed hi))."""
    q = np.arange((V + 3) // 4, dtype=np.uint64)
    words = philox4x32_10(q, step, img, sample, seed & 0xFFFFFFFF, seed >> 32)
    return np.stack(words, axis=1).reshape(-1)[:V]


def gumbel(bits):
    """fp64 Gumbel noise of Philox words: u = ((bits >> 8) + 0.5) * 2^-24 in (0, 1), g = -log(-log(u))."""
    u = ((bits >> 8).astype(np.float64) + 0.5) * 2.0 ** -24
    return -np.log(-np.log(u))


def candidates(l, top_k):
    """Candidate ids: every token for top_k 0 (or V), else the top_k largest l, ties to the lower id."""
    V = l.shape[0]
    if top_k == 0 or top_k >= V:
        return np.arange(V)
    order = np.lexsort((np.arange(V), -l))                  # l descending, then id ascending
    return np.sort(order[:top_k])


def select(logits, temperature, top_k, seed, step, img, sample):
    """One draw from the logits (V,) of a step -> (token, lp, margin).  lp = log_softmax(logits)[token] in the logits' dtype.
    margin: how far the draw is from changing — greedy: the top-2 gap of l; Gumbel: the gap between the two largest keys,
    and with a top-k restriction also the gap at the top-k boundary (l sorted, k-th minus (k+1)-th)."""
    l = logits.detach().double().cpu().numpy()
    V = l.shape[0]
    lp_all = F.log_softmax(logits, dim=0)
    if temperature == 0:
        tok = int(np.argmax(l))                              # first maximum: the lowest id
        s = np.sort(l)[::-1]
        margin = float(s[0] - s[1]) if V > 1 else float("inf")
        return tok, lp_all[tok], margin
    cand = candidates(l, top_k)
    key = l[cand] / temperature + gumbel(token_bits(seed, step, img, sample, V))[cand]
    best = int(np.argmax(key))
    tok = int(cand[best])
    ks = np.sort(key)[::-1]
    margin = float(ks[0] - ks[1]) if len(ks) > 1 else float("inf")
    if 0 < top_k < V:
        s = np.sort(l)[::-1]
        margin = min(margin, float(s[top_k - 1] - s[top_k]))
    return tok, lp_all[tok], margin


def sample_image(step_fn, state, m, start_id, end_id, max_steps, temperature, top_k, seed, img, sample_base=0):
    """The m samples of one image.  ``state``: the start state of one row (tuple of tensors with first dim 1);
    ``step_fn(state, prev_words (1, 1)) -> (logits (1, V), state)``.  Each sample runs steps 1 .. max_steps+1 from that state
    (step 1 is the same computation for every sample).  Returns per sample a dict: seq, len, ended, score (summed in the
    logits' dtype, step order), logp (list), margins (list, one per step)."""
    out = []
    for j in range(m):
        st, prev = state, start_id
        seq, logp, margins = [start_id], [], []
        score = None
        ended = False
        for step in range(1, max_steps + 2):
            logits, st = step_fn(st, torch.tensor([[prev]], dtype=torch.long))
            tok, lp, mg = select(logits[0], temperature, top_k, seed, step, img, sample_base + j)
            score = lp if score is None else score + lp
            seq.append(tok); logp.append(float(lp)); margins.append(mg)
            prev = tok
            if tok == end_id:
                ended = True
                break
        out.append(dict(seq=seq, len=len(seq), ended=ended, score=float(score), logp=logp, margins=margins))
    return out


def baseline_start(w, img_features):
    """(step_fn, start state) of the BaselineDecoder as ``baseline_beam_reference.baseline_beam_search`` builds them: the image
    feature is an unscored step 0 from the zero state, then emb(previous word) per step."""
    dtype = w["linear.weight"].dtype
    H = w["lstm.weight_hh_l0"].size(1)
    cell = (w["lstm.weight_ih_l0"], w["lstm.weight_hh_l0"], w["lstm.bias_ih_l0"], w["lstm.bias_hh_l0"])
    zero = torch.zeros(1, H, dtype=dtype)
    h0, c0 = lstm_cell(img_features.reshape(1, -1).to(dtype), zero, zero, *cell)

    def step(state, prev):
        h, c = state
        x = F.embedding(prev, w["embedding.weight"]).squeeze(1).to(dtype)
        h, c = lstm_cell(x, h, c, *cell)
        return F.linear(h, w["linear.weight"], w["linear.bias"]), (h, c)

    return step, (h0, c0)


def attention_start(w, encoder_out):
    """(step_fn, start state) of the attention decoder: ``baseline_beam_reference.attention_step`` from init_hidden_state."""
    step, enc = BR.attention_step(w, encoder_out)
    h, c = init_hidden_state(w, enc)
    return step, (enc, h, c)
