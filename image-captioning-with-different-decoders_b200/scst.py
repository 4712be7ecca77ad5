"""Self-critical sequence training (SCST) for both decoders, built on ``gen_captions.sample_captions``.

One call of ``self_critical_loss`` (the definition is restated on the CPU in tests/scst_reference.py):
1. draws ``n_samples`` captions per image with the sampler (no gradient) and scores them with the caller's ``reward_fn``;
2. forms the advantage ``A = r - b`` against a baseline ``b``: the reward of the greedy caption ("greedy", the self-critical
   baseline) or the mean reward of the image's other samples ("mean", leave-one-out);
3. packs the samples as one training batch, rows sorted by length (``pack_samples``), and runs the decoder's training forward
   on them in eval mode (the sampled distribution has no dropout); the attention decoder reads each image's features once
   for its m rows (``forward(..., image_index=)``), the baseline decoder gets its (E,) feature replicated per row;
4. returns ``(1/N) sum A_row * CE(logits, next token)`` over the N scored tokens — ``-(1/N) sum A * logp`` — formed by the
   weighted fused cross-entropy kernels (``losses.weighted_token_loss``).
The scored positions are exactly the sampler's steps 1 .. len-1, ``<end>`` included when it was drawn.  In the fp32 and
fp32x3 tiers the forward's log-probabilities equal the sampler's up to the tier's rounding; the attention decoder's bf16
training tier evaluates them with bf16 operands, so its gradient is slightly off-policy (DESIGN.md section 5.6 gives the
measured gap).
"""
import numpy as np
import torch

from . import _lib
from .gen_captions import sample_captions
from .losses import packed_targets, weighted_token_loss
from .models.baseline import BaselineDecoder


class PackedSamples:
    """The n x m samples of ``sample_captions`` as R = n*m training rows, sorted by a stable descending sort of the length
    (ties keep the flat index i*m + j), as the attention forward needs (it runs the first ``batch_size_t`` rows)."""

    def __init__(self, captions, lengths, img_idx, perm, n, m, img_idx_host=None):
        self.captions = captions      # (R, Lmax) int64, 0 beyond the length
        self.lengths = lengths        # list of R ints
        self.img_idx = img_idx        # (R,) int64: image of each row
        self.img_idx_host = img_idx_host   # the same on the CPU (the attention forward's image_index: no device round trip)
        self.perm = perm              # (R,) int64: flat index i*m + j of each row
        self.n, self.m = n, m

    def pack(self, x):
        """(n, m, ...) per-sample values -> (R, ...) in row order."""
        return x.reshape(self.n * self.m, *x.shape[2:])[self.perm.to(x.device)]

    def unpack(self, x):
        """(R, ...) per-row values -> (n, m, ...), the inverse of ``pack``."""
        out = torch.empty_like(x)
        out[self.perm.to(x.device)] = x
        return out.reshape(self.n, self.m, *x.shape[1:])


def pack_samples(samples):
    """``samples``: a dict with ``seq`` (n, m, S) and ``len`` (n, m) as ``sample_captions`` returns them -> PackedSamples."""
    seq, ln = samples["seq"], samples["len"]
    n, m = ln.shape
    flat_len = ln.reshape(-1).cpu().numpy().astype(np.int64)
    order = np.argsort(-flat_len, kind="stable")
    lengths = flat_len[order].tolist()
    Lmax = lengths[0]
    dev = seq.device
    perm = torch.from_numpy(order).to(dev)
    rows = seq.reshape(n * m, -1)[perm, :Lmax].long()
    keep = torch.arange(Lmax, device=dev)[None, :] < torch.tensor(lengths, device=dev)[:, None]
    captions = torch.where(keep, rows, torch.zeros_like(rows))
    return PackedSamples(captions, lengths, perm // m, perm, n, m, torch.from_numpy(order // m))


def scored_targets(captions, lengths, baseline_decoder, row_valid=None):
    """The training targets of packed samples, -1 at unscored positions.  Attention decoder: (R, Lmax-1), position t < len-1
    predicts captions[:, t+1] (``losses.packed_targets``; ``row_valid`` is the forward's activity mask).  Baseline decoder:
    (R, Lmax), positions 1 <= t <= len-1 predict captions[:, t]; position 0 is the unscored image step."""
    if not baseline_decoder:
        Lm1 = captions.shape[1] - 1
        return packed_targets(captions, [l - 1 for l in lengths], Lm1, row_valid)[0]
    t = torch.arange(captions.shape[1], device=captions.device)[None, :]
    ln = torch.tensor(lengths, device=captions.device)[:, None]
    return torch.where((t >= 1) & (t < ln), captions, torch.full_like(captions, -1))


def baseline_rewards(rewards, kind, greedy_rewards=None):
    """b of the advantage A = r - b for (n, m) rewards.  "greedy": the (n,) rewards of the greedy captions, broadcast over the
    m samples; "mean" (leave-one-out): b_ij = (sum_k r_ik - r_ij) / (m - 1), m >= 2."""
    n, m = rewards.shape
    if kind == "greedy":
        return greedy_rewards.reshape(n, 1).expand(n, m).contiguous()
    if m < 2:
        raise ValueError("baseline='mean' (leave-one-out) needs n_samples >= 2")
    return (rewards.sum(dim=1, keepdim=True) - rewards) / (m - 1)


def _rewards(reward_fn, seq, ln, shape):
    r = reward_fn(seq, ln)
    if not isinstance(r, torch.Tensor) or not r.is_floating_point() or tuple(r.shape) != shape or not r.is_cuda:
        raise ValueError("reward_fn must return a %s floating-point CUDA tensor, got %s" %
                         (shape, tuple(r.shape) if isinstance(r, torch.Tensor) else type(r).__name__))
    r = r.float()
    if not bool(torch.isfinite(r).all()):
        raise ValueError("reward_fn returned a non-finite reward")
    return r


def self_critical_loss(decoder, features, reward_fn, n_samples, start_id, end_id, baseline="greedy", temperature=1.0,
                       top_k=0, seed=None, max_steps=50, sample_precision="fp32x3", bf16_grad_only=False):
    """One SCST loss of an ``AttentionDecoder`` (features as ``beam_search_batched`` takes them) or a ``BaselineDecoder``
    ((n, E) image features).  ``reward_fn(seq, len)`` gets the sampler's (n, m, max_steps+2) int32 captions and (n, m) lengths
    and returns (n, m) floating-point CUDA rewards.  The samples are drawn by ``sample_captions`` with ``temperature``,
    ``top_k``, ``seed`` and ``max_steps`` in ``sample_precision`` ("fp32x3" or "fp32"); the training forward and backward run in
    ``decoder.precision``.  ``bf16_grad_only``: as in ``attention_caption_loss`` (attention decoder, bf16 tier).
    -> (loss, info): ``loss`` a 0-dim tensor whose graph reaches the decoder parameters (and ``features`` when they require a
    gradient: summed over the samples of each image); ``info`` holds seq, len, ended, seed (the sampler's), rewards, baseline,
    advantages ((n, m) fp32), n_tokens (N) and logp: the forward's log-probability of every scored token in the sampler's
    (n, m, max_steps+1) layout (0 beyond len-1)."""
    if baseline not in ("greedy", "mean"):
        raise ValueError("baseline must be 'greedy' or 'mean'")
    m = int(n_samples)
    if m < 1:
        raise ValueError("n_samples must be >= 1")
    if baseline == "mean" and m < 2:
        raise ValueError("baseline='mean' (leave-one-out) needs n_samples >= 2")
    if sample_precision not in ("fp32", "fp32x3"):
        raise ValueError("caption sampling runs in fp32-grade arithmetic only: sample_precision must be 'fp32' or 'fp32x3'")
    if not features.is_cuda:
        raise _lib.IcdError("self_critical_loss needs CUDA tensors; there is no CPU fallback")
    n = features.shape[0]
    base = isinstance(decoder, BaselineDecoder)
    with torch.no_grad():
        s = sample_captions(decoder, features.detach(), m, start_id, end_id, temperature=temperature, top_k=top_k, seed=seed,
                            max_steps=max_steps, want_logp=True, precision=sample_precision)
        r = _rewards(reward_fn, s["seq"], s["len"], (n, m))
        gr = None
        if baseline == "greedy":
            g = sample_captions(decoder, features.detach(), 1, start_id, end_id, temperature=0.0, seed=s["seed"],
                                max_steps=max_steps, precision=sample_precision)
            gr = _rewards(reward_fn, g["seq"], g["len"], (n, 1))[:, 0]
        b = baseline_rewards(r, baseline, gr)
        adv = r - b
    pk = pack_samples(s)
    R = n * m
    lengths = pk.lengths
    n_tokens = sum(lengths) - R
    was_training = decoder.training
    decoder.eval()
    try:
        if base:
            logits = decoder(features[pk.img_idx], pk.captions)
        else:
            logits = decoder(features, pk.captions, lengths, image_index=pk.img_idx_host)[0]
        tgt = scored_targets(pk.captions, lengths, base, getattr(logits, "_icd_row_valid", None))
        w = pk.pack(adv)[:, None].expand(R, logits.shape[1]).contiguous()
        loss = weighted_token_loss(logits, tgt, w, n_tokens, bf16_grad_only=bf16_grad_only)
    finally:
        decoder.train(was_training)
    row_lp = (0.0 - loss.row_loss).view(R, -1)
    if base:
        row_lp = row_lp[:, 1:]                     # position 0 is the unscored image step
    lp = torch.zeros(R, max_steps + 1, device=row_lp.device, dtype=torch.float32)
    lp[:, :row_lp.shape[1]] = row_lp
    info = dict(seq=s["seq"], len=s["len"], ended=s["ended"], seed=s["seed"], rewards=r, baseline=b, advantages=adv,
                n_tokens=n_tokens, logp=pk.unpack(lp))
    return loss, info
