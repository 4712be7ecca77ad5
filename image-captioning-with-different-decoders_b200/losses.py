"""Loss glue of the reference train loops as fused kernels (SURVEY.md 8f rank 1).

``attention_caption_loss`` == models/attention.py:401-414:

    targets = captions[:, 1:]
    scores  = pack_padded_sequence(scores,  decode_lengths, batch_first=True).data
    targets = pack_padded_sequence(targets, decode_lengths, batch_first=True).data
    loss = CrossEntropyLoss()(scores, targets) + ((alpha_c - alphas.sum(dim=1)) ** 2).mean()

The mean cross-entropy over the packed rows does not depend on their order, so the 466 MB packed copy and the
separate log-softmax / NLL / softmax-backward passes are replaced by two streaming kernels (icd_cross_entropy_fwd:
per-row loss + log-sum-exp; icd_cross_entropy_bwd: gradient, scaled by the upstream gradient read on the device, plus
a bf16 copy for the tensor-core tier); rows with t >= batch_size_t carry target -1 and are skipped
(they are the rows pack_padded_sequence drops).  ``baseline_caption_loss`` == models/baseline.py:194-195,224-225
(CrossEntropyLoss(ignore_index=<pad>) over all (b, t)).
The doubly-stochastic regulariser over the (B,T,196) alphas is one forward and one backward kernel (``alpha_regulariser``).
"""
import numpy as np
import torch

from . import ops


# bf16 hand-off between the fused loss and the bf16 tier of the decoder backward: the loss backward already streams every
# logit once, so it also emits the bf16 copy of d(loss)/d(logits) that the vocabulary-layer backward contractions consume —
# the decoder backward then skips its own fp32 -> bf16 pass over the (B*T, V) gradient.  The copy travels in a small box
# that belongs to ONE decoder forward: the decoder's autograd node and the `predictions` tensor it returned both hold it
# (`predictions._icd_box`), the loss stores it in its own node, so two decoder / loss pairs in one graph (micro-batches,
# two models) never see each other's gradient, nothing is process-global, and the box dies with the graph.
class GradBox:
    """Per-decoder-forward mailbox: filled by _FusedCE.backward, emptied by the decoder backward."""
    __slots__ = ("d16", "d32", "version", "hollow", "hollow_expected")

    def __init__(self):
        self.d16 = self.d32 = None
        self.version = -1
        self.hollow = False              # the fp32 gradient that was sent is hollow (bf16_grad_only=True)
        self.hollow_expected = False     # a bf16_grad_only loss was built on this forward: fp32 d_predictions is NOT to be trusted

    def put(self, d16, d32, hollow):
        self.d16, self.d32, self.version, self.hollow = d16, d32, d32._version, hollow

    def take(self, grad):
        """-> the bf16 gradient matching the fp32 tensor ``grad`` that reached the decoder backward, or None when the
        loss produced none.  Raises when only a HOLLOW fp32 gradient exists and it is not exactly what arrived (autograd
        summed it with another gradient, or something modified it in place) — never reads undefined memory."""
        d16, d32, version, hollow = self.d16, self.d32, self.version, self.hollow
        self.d16 = self.d32 = None
        ok = (d16 is not None and d32 is not None and d32.data_ptr() == grad.data_ptr() and d32.numel() == grad.numel()
              and d32._version == version and grad._version == version)
        if ok:
            return d16
        if hollow or self.hollow_expected:
            raise RuntimeError("attention_caption_loss(bf16_grad_only=True): the logit gradient reaching the decoder is not "
                               "the one the loss produced (predictions feed something else too, or the gradient was "
                               "modified on its way); use bf16_grad_only=False")
        return None


_FUSED_CE_MAX_V = 49000          # rows up to this many classes fit the one-pass kernel's shared memory (icd_cross_entropy_fwd_grad16)


class _FusedCE(torch.autograd.Function):
    """sum_r weights[r] * CE_r / n_valid over the rows with target >= 0; ``weights`` None is the plain mean (every weight 1)."""

    @staticmethod
    def forward(ctx, logits2d, targets, n_valid, want_bf16, bf16_only=False, box=None, weights=None):
        ctx.n_valid, ctx.want_bf16 = n_valid, bool(want_bf16 and box is not None)
        ctx.bf16_only = bool(bf16_only and ctx.want_bf16)
        ctx.box = box
        ctx.d16 = None
        if ctx.bf16_only and ctx.needs_input_grad[0] and logits2d.shape[1] <= _FUSED_CE_MAX_V:
            # training fast path: the only gradient anyone will ask for is the bf16 one, so it is formed in the SAME pass over
            # the logits as the loss (each row parked in shared memory); the backward only applies the upstream scalar
            row_loss, lse, ctx.d16 = ops.cross_entropy_fwd_grad16(logits2d, targets, 1.0 / n_valid, weights=weights)
        else:
            row_loss, lse = ops.cross_entropy_fwd(logits2d, targets)
        ctx.save_for_backward(logits2d, targets, lse, weights)
        if ctx.bf16_only:
            box.hollow_expected = True
        if weights is None:
            return row_loss.sum() / n_valid
        out = (row_loss * weights).sum() / n_valid
        out.row_loss = row_loss                      # per-row unweighted cross-entropy (weighted_token_loss documents it)
        return out

    @staticmethod
    def backward(ctx, g):
        logits2d, targets, lse, weights = ctx.saved_tensors
        g = g.reshape(1).float().contiguous()
        if ctx.d16 is not None:
            d16, ctx.d16 = ops.scale_bf16_by_device_scalar(ctx.d16, g), None
            d_logits = torch.empty_like(logits2d)            # hollow: never written, never read (GradBox refuses anything else)
            ctx.box.put(d16, d_logits, True)
            return d_logits, None, None, None, None, None, None
        d_logits, d16 = ops.cross_entropy_bwd(logits2d, targets, lse, 1.0 / ctx.n_valid, upstream=g,
                                              want_bf16=ctx.want_bf16, want_fp32=not ctx.bf16_only, weights=weights)
        if d16 is not None:
            ctx.box.put(d16, d_logits, ctx.bf16_only)
        return d_logits, None, None, None, None, None, None


class _AlphaReg(torch.autograd.Function):
    """((alpha_c - alphas.sum(dim=1)) ** 2).mean() as one forward and one backward kernel (the torch expression is eight)."""

    @staticmethod
    def forward(ctx, alphas, alpha_c):
        reg, resid = ops.alpha_regulariser_fwd(alphas, alpha_c)
        ctx.save_for_backward(resid)
        ctx.T = alphas.shape[1]
        return reg

    @staticmethod
    def backward(ctx, g):
        (resid,) = ctx.saved_tensors
        return ops.alpha_regulariser_bwd(resid, ctx.T, upstream=g.reshape(1).float().contiguous()), None


def alpha_regulariser(alphas, alpha_c=1.0):
    """Doubly stochastic attention regulariser of models/attention.py:413-414."""
    return _AlphaReg.apply(alphas.float().contiguous(), float(alpha_c))        # CUDA only, like every op of this package


def packed_targets(encoded_captions, decode_lengths, T, row_valid=None):
    """targets[b, t] = captions[b, t+1] where row b is active at step t (b < batch_size_t), else -1.
    ``row_valid``: the (B*T) uint8 activity mask the decoder forward already built on the device (no host->device
    copy, no sync); rebuilt from ``decode_lengths`` when absent."""
    B = encoded_captions.shape[0]
    dev = encoded_captions.device
    if row_valid is not None:
        active = row_valid.view(B, T).bool()
    else:
        dl = np.asarray(decode_lengths, dtype=np.int64)
        bt = (dl[None, :] > np.arange(T)[:, None]).sum(axis=1)                       # batch_size_t
        active = torch.from_numpy(np.arange(B)[:, None] < bt[None, :]).to(dev, non_blocking=True)
    tgt = encoded_captions[:, 1:T + 1]
    return torch.where(active, tgt, torch.full_like(tgt, -1)), int(sum(decode_lengths))


def _dp_token_scale(n_valid, device, group=None):
    """n_local * world / n_global as a DEVICE scalar (one tiny all-reduce, no host sync): with it the mean over ranks of the
    per-rank mean losses is the mean over ALL packed tokens, i.e. the reference's single-process (N*B)-caption step, also
    when the ranks hold different numbers of packed tokens (ragged COCO batches).  Exactly 1 for equal-length batches."""
    import torch.distributed as dist
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        return None
    cnt = torch.tensor([float(n_valid)], device=device, dtype=torch.float64)
    dist.all_reduce(cnt, op=dist.ReduceOp.SUM, group=group)
    return (float(n_valid) * dist.get_world_size(group) / cnt).float().reshape(())


def attention_caption_loss(predictions, encoded_captions, decode_lengths, alphas, alpha_c=1.0, bf16_grad_only=False,
                           dp_token_weighting=False, dp_group=None):
    """bf16_grad_only (bf16 tier only): the loss backward writes ONLY the bf16 copy of d(loss)/d(logits) that the decoder
    backward consumes and leaves the 466 MB fp32 gradient tensor hollow.  Valid when ``predictions`` feeds nothing but this
    loss in the autograd graph — the reference train loop (models/attention.py:401-414; its top-5 accuracy is computed
    without a graph).  If the gradient is modified on its way to the decoder the backward raises instead of reading it.
    dp_token_weighting (data parallel, ragged batches): weight this rank's cross-entropy by n_local * world / n_global so
    that the 1/world-averaged gradient equals the single-process big-batch gradient (see _dp_token_scale)."""
    B, T, V = predictions.shape
    tgt, n_valid = packed_targets(encoded_captions, decode_lengths, T, getattr(predictions, "_icd_row_valid", None))
    box = getattr(predictions, "_icd_box", None)
    want_bf16 = bool(getattr(predictions, "_icd_bf16_tier", False)) and box is not None
    ce = _FusedCE.apply(predictions.reshape(B * T, V), tgt.reshape(-1).contiguous(), n_valid, want_bf16, bf16_grad_only, box)
    if dp_token_weighting:
        scale = _dp_token_scale(n_valid, predictions.device, dp_group)
        if scale is not None:
            ce = ce * scale
    return ce + alpha_regulariser(alphas, alpha_c)


def weighted_token_loss(logits, targets, weights, count, bf16_grad_only=False):
    """sum over the scored positions of weights * cross-entropy, divided by ``count`` — the token loss of sequence-level
    training (scst.self_critical_loss: the weight of a token is its caption's advantage).  ``logits`` (B, T, V) from either
    decoder's forward; ``targets`` (B, T) int64, -1 at unscored positions; ``weights`` (B, T) fp32 (no gradient flows to
    them; any sign); ``count`` a host number.  The gradient is formed by the weighted fused kernels
    (icd_weighted_cross_entropy_bwd / _fwd_grad16) and, from the attention decoder's bf16 tier, handed to the decoder
    backward as bf16 like ``attention_caption_loss`` does; ``bf16_grad_only`` has the same meaning and conditions there.
    The result carries ``.row_loss``: the (B*T,) unweighted cross-entropy of every position (0 where the target is -1),
    i.e. -log p of each scored token, with no gradient."""
    B, T, V = logits.shape
    assert targets.shape == (B, T) and weights.shape == (B, T), "targets and weights must be (B, T) like the logits"
    box = getattr(logits, "_icd_box", None)
    want_bf16 = bool(getattr(logits, "_icd_bf16_tier", False)) and box is not None
    w = weights.detach().to(device=logits.device, dtype=torch.float32).reshape(-1).contiguous()
    return _FusedCE.apply(logits.reshape(B * T, V), targets.reshape(-1).contiguous(), count, want_bf16, bf16_grad_only, box, w)


class _MaskedMeanCE(torch.autograd.Function):
    """mean over the rows with target >= 0 of the row cross-entropy, the count staying ON THE DEVICE (no host sync):
    forward = sum(row_loss) / count; backward scales the upstream gradient by 1 / count before the streaming kernel."""

    @staticmethod
    def forward(ctx, logits2d, targets):
        row_loss, lse = ops.cross_entropy_fwd(logits2d, targets)
        inv = 1.0 / (targets >= 0).sum().clamp_min(1).float()
        ctx.save_for_backward(logits2d, targets, lse, inv)
        return row_loss.sum() * inv

    @staticmethod
    def backward(ctx, g):
        logits2d, targets, lse, inv = ctx.saved_tensors
        up = (g.reshape(1).float() * inv).contiguous()
        return ops.cross_entropy_bwd(logits2d, targets, lse, 1.0, upstream=up)[0], None


def baseline_caption_loss(outputs, captions, pad_id=0):
    """CrossEntropyLoss(ignore_index=<pad>)(scores.reshape(-1, V), captions.reshape(-1)) — models/baseline.py:194-195,
    224-225 — as the two streaming kernels; the number of non-pad targets never leaves the device."""
    B, L, V = outputs.shape
    tgt = torch.where(captions == pad_id, torch.full_like(captions, -1), captions).reshape(-1).contiguous()
    return _MaskedMeanCE.apply(outputs.reshape(B * L, V), tgt)
