"""Caption generation with beam search — drop-in for gen_captions.py:16-131, plus a batched entry point.

``attention_caption_image_beam_search(device, args, img, encoder, decoder, vocab)`` keeps the reference signature
and return tuple ``(seq, alphas, Caption_End)``; ``beam_search_batched`` decodes many images at once with the
device-side engine of ``icd_beam_search`` (csrc/beam.cu): no per-step host synchronisation, features indexed per
image, ``enc_att`` computed once per image.

The reference has no generation function for the ``BaselineDecoder``.  ``baseline_beam_search_batched`` and
``baseline_caption_image_beam_search`` give it one (``icd_baseline_beam_search``): the same beam state machine over the
baseline's step.  The image feature is LSTM step 0 from the zero state and its logits are not scored: teacher forcing
trains ``outputs[:, 0]`` against ``captions[:, 0] = <start>`` (models/baseline.py:93-109), so position 0 of every
caption is ``<start>`` and the first scored prediction is conditioned on ``emb(<start>)``.  ``beam_size = 1`` is
greedy decoding.

``sample_captions`` draws captions at random from either decoder instead (seeded temperature / top-k sampling,
``icd_sample_captions`` / ``icd_baseline_sample_captions``), with the log-probability of every sampled token.
"""
import ctypes

import torch

from . import _lib, ops
from ._lib import check, fill, lib, stream_ptr
from .models.baseline import BaselineDecoder
from .vocabulary import END_TOKEN, START_TOKEN


def beam_search_batched(decoder, features, beam_size, start_id, end_id, max_steps=50,
                        want_alphas=True, want_trace=False, chunk=None, precision="fp32x3"):
    """features (n_img, 14, 14, C) or (n_img, P, C) CUDA fp32 -> dict with
         len    (n_img,) int32  caption length incl. <start>/<end>; 0 = no beam completed (reference failure tuple)
         seq    (n_img, max_steps+2) int32
         score  (n_img,) float32 raw summed log-prob of the winner (gen_captions.py:127)
         alpha  (n_img, max_steps+2, P) float32, frame 0 all ones (gen_captions.py:54)      [want_alphas]
         trace  (max_steps+1, n_img, k) int32 next-word ids per step, -1 = empty slot        [want_trace]
    The loop body runs for step = 1 .. max_steps+1, like ``step > 50`` at gen_captions.py:119 for max_steps=50.
    Caption generation needs fp32-grade logits for identical captions (SURVEY.md 7.2): ``precision`` is "fp32x3" (default:
    3-term bf16 split on the tcgen05 tensor cores, ~6e-6 relative) or "fp32" (fp32 FMA kernel); never "bf16"."""
    if precision not in ("fp32", "fp32x3"):
        raise ValueError("beam search runs in fp32-grade arithmetic only: precision must be 'fp32' or 'fp32x3'")
    if not features.is_cuda:
        raise _lib.IcdError("beam_search_batched needs CUDA tensors; there is no CPU fallback")
    n_img = features.shape[0]
    C = features.shape[-1]
    enc = features.reshape(n_img, -1, C).contiguous().float()
    P = enc.shape[1]
    k = int(beam_size)
    dev = enc.device
    a = decoder.attention
    A, D, E, V = a.enc_att.weight.shape[0], decoder.decode_step.weight_hh.shape[1], \
        decoder.embedding.weight.shape[1], decoder.fc.weight.shape[0]
    if chunk is None:
        chunk = max(1, min(n_img, 65535 // k))
    S2 = max_steps + 2
    out = dict(len=torch.empty(n_img, device=dev, dtype=torch.int32),
               seq=torch.zeros(n_img, S2, device=dev, dtype=torch.int32),
               score=torch.empty(n_img, device=dev, dtype=torch.float32))
    if want_alphas:
        out["alpha"] = torch.zeros(n_img, S2, P, device=dev, dtype=torch.float32)
    traces = []
    emb_w = decoder.embedding.weight
    ws_cache = None
    for i0 in range(0, n_img, chunk):
        n = min(chunk, n_img - i0)
        d = _lib.BeamDesc()
        trace = torch.empty(max_steps + 1, n, k, device=dev, dtype=torch.int32) if want_trace else None
        fill(d, n_img=n, k=k, max_steps=max_steps, P=P, C=C, A=A, D=D, E=E, V=V,
             precision=ops.precision_id(precision), emb_is_f64=int(emb_w.dtype == torch.float64),
             start_id=start_id, end_id=end_id, enc=enc[i0:i0 + n],
             enc_att_w=a.enc_att.weight, enc_att_b=a.enc_att.bias, dec_att_w=a.dec_att.weight,
             dec_att_b=a.dec_att.bias, full_att_w=a.full_att.weight, full_att_b=a.full_att.bias,
             w_ih=decoder.decode_step.weight_ih, w_hh=decoder.decode_step.weight_hh,
             b_ih=decoder.decode_step.bias_ih, b_hh=decoder.decode_step.bias_hh,
             h_lin_w=decoder.h_lin.weight, h_lin_b=decoder.h_lin.bias, c_lin_w=decoder.c_lin.weight,
             c_lin_b=decoder.c_lin.bias, f_beta_w=decoder.f_beta.weight, f_beta_b=decoder.f_beta.bias,
             fc_w=decoder.fc.weight, fc_b=decoder.fc.bias, emb_w=emb_w,
             out_len=out["len"][i0:i0 + n], out_seq=out["seq"][i0:i0 + n], out_score=out["score"][i0:i0 + n],
             out_alpha=(out["alpha"][i0:i0 + n] if want_alphas else None), trace_words=trace)
        need = int(lib().icd_beam_search_ws_bytes(ctypes.byref(d)))
        if ws_cache is None or ws_cache.numel() < need:
            ws_cache = torch.empty(need, device=dev, dtype=torch.uint8)
        d.ws = ws_cache.data_ptr()
        d.ws_bytes = need
        check(lib().icd_beam_search(ctypes.byref(d), stream_ptr()), "icd_beam_search")
        if want_trace:
            traces.append(trace)
    if want_trace:
        out["trace"] = torch.cat(traces, dim=1)
    return out


def baseline_beam_search_batched(decoder, img_features, beam_size, start_id, end_id, max_steps=50, want_trace=False,
                                 chunk=None, precision="fp32x3"):
    """Beam search over a ``BaselineDecoder``.  img_features (n_img, E) CUDA — what the baseline encoder returns; cast to
    fp32 like the forward does (models/baseline.py:101) -> dict with
         len    (n_img,) int32  caption length incl. <start>/<end>; 0 = no beam completed (failure)
         seq    (n_img, max_steps+2) int32, seq[:, 0] = <start>
         score  (n_img,) float32 raw summed log-prob of the winner over steps 1 .. len-1
         trace  (max_steps+1, n_img, k) int32 next-word ids per step, -1 = empty slot        [want_trace]
    Step 0 feeds the image feature from the zero LSTM state and is not scored; steps 1 .. max_steps+1 feed emb(previous
    word), <start> at step 1, with the state machine of ``beam_search_batched`` (gen_captions.py:16-131).  ``beam_size``
    1 is greedy decoding.  ``precision`` is "fp32x3" (default) or "fp32"; never "bf16": identical captions need
    fp32-grade logits.  An fp64 (GloVe) embedding table is cast to fp32 once per call."""
    if precision not in ("fp32", "fp32x3"):
        raise ValueError("beam search runs in fp32-grade arithmetic only: precision must be 'fp32' or 'fp32x3'")
    if not img_features.is_cuda:
        raise _lib.IcdError("baseline_beam_search_batched needs CUDA tensors; there is no CPU fallback")
    img = img_features.contiguous().float()
    n_img, E = img.shape
    k = int(beam_size)
    dev = img.device
    lstm, lin = decoder.lstm, decoder.linear
    ws = [t.detach().contiguous() for t in (lstm.weight_ih_l0, lstm.weight_hh_l0, lstm.bias_ih_l0, lstm.bias_hh_l0,
                                             lin.weight, lin.bias)]
    emb_w = decoder.embedding.weight.detach().contiguous()
    H, V = ws[1].shape[1], ws[4].shape[0]
    assert emb_w.shape[1] == E, "img_features must have the embedding width %d" % emb_w.shape[1]
    if chunk is None:
        chunk = max(1, min(n_img, 65535 // k))
    S2 = max_steps + 2
    out = dict(len=torch.empty(n_img, device=dev, dtype=torch.int32),
               seq=torch.zeros(n_img, S2, device=dev, dtype=torch.int32),
               score=torch.empty(n_img, device=dev, dtype=torch.float32))
    traces = []
    ws_cache = None
    for i0 in range(0, n_img, chunk):
        n = min(chunk, n_img - i0)
        d = _lib.BaseBeamDesc()
        trace = torch.empty(max_steps + 1, n, k, device=dev, dtype=torch.int32) if want_trace else None
        fill(d, n_img=n, k=k, max_steps=max_steps, E=E, H=H, V=V, precision=ops.precision_id(precision),
             emb_is_f64=int(emb_w.dtype == torch.float64), start_id=start_id, end_id=end_id, img_features=img[i0:i0 + n],
             emb_w=emb_w, w_ih=ws[0], w_hh=ws[1], b_ih=ws[2], b_hh=ws[3], lin_w=ws[4], lin_b=ws[5],
             out_len=out["len"][i0:i0 + n], out_seq=out["seq"][i0:i0 + n], out_score=out["score"][i0:i0 + n],
             trace_words=trace)
        need = int(lib().icd_baseline_beam_search_ws_bytes(ctypes.byref(d)))
        if ws_cache is None or ws_cache.numel() < need:
            ws_cache = torch.empty(need, device=dev, dtype=torch.uint8)
        d.ws = ws_cache.data_ptr()
        d.ws_bytes = need
        check(lib().icd_baseline_beam_search(ctypes.byref(d), stream_ptr()), "icd_baseline_beam_search")
        if want_trace:
            traces.append(trace)
    if want_trace:
        out["trace"] = torch.cat(traces, dim=1)
    return out


def sample_captions(decoder, features, n_samples, start_id, end_id, temperature=1.0, top_k=0, seed=None, max_steps=50,
                    want_logp=False, chunk=None, precision="fp32x3", sample_base=0):
    """Draw ``n_samples`` captions per image from an ``AttentionDecoder`` (features as for ``beam_search_batched``) or a
    ``BaselineDecoder`` (img_features as for ``baseline_beam_search_batched``) -> dict with
         seq    (n_img, n_samples, max_steps+2) int32, seq[..., 0] = <start>, 0 beyond len
         len    (n_img, n_samples) int32  length incl. <start> and <end>; max_steps+2 for a truncated sample
         ended  (n_img, n_samples) uint8  1 = the sample drew <end>, 0 = truncated after step max_steps+1
         score  (n_img, n_samples) float32 sum of the log-probabilities of the sampled tokens (steps 1 .. len-1)
         logp   (n_img, n_samples, max_steps+1) float32 each step's term, 0 beyond len-1          [want_logp]
         seed   the seed used
    Every step draws from softmax(logits / temperature) restricted to the ``top_k`` largest logits (0: all) by Gumbel-max
    with counter-based noise keyed by (seed, image index, sample index, step, token); ``temperature = 0`` is greedy.  The
    log-probabilities are those of the model at temperature 1 over the whole vocabulary.  Sample j of an image is the same
    whatever ``chunk`` is, whichever images share the call and however many samples are drawn; ``sample_base`` is the
    global index of the first sample (more samples of the same images later: the next indices).  ``seed=None`` draws one
    from torch's default CPU generator (``torch.manual_seed`` makes runs reproducible).  ``precision`` is "fp32x3" or "fp32";
    never "bf16"."""
    if precision not in ("fp32", "fp32x3"):
        raise ValueError("caption sampling runs in fp32-grade arithmetic only: precision must be 'fp32' or 'fp32x3'")
    if not features.is_cuda:
        raise _lib.IcdError("sample_captions needs CUDA tensors; there is no CPU fallback")
    n = int(n_samples)
    if n < 1:
        raise ValueError("n_samples must be >= 1")
    if seed is None:
        seed = int(torch.randint(0, 2 ** 63 - 1, (1,), dtype=torch.int64).item())
    seed = int(seed) & (2 ** 64 - 1)
    base = isinstance(decoder, BaselineDecoder)
    n_img = features.shape[0]
    dev = features.device
    if base:
        x = features.contiguous().float()
        lstm, lin = decoder.lstm, decoder.linear
        ws = [t.detach().contiguous() for t in (lstm.weight_ih_l0, lstm.weight_hh_l0, lstm.bias_ih_l0, lstm.bias_hh_l0,
                                                 lin.weight, lin.bias)]
        emb_w = decoder.embedding.weight.detach().contiguous()
        E = x.shape[1]
        H, V = ws[1].shape[1], ws[4].shape[0]
        assert emb_w.shape[1] == E, "img_features must have the embedding width %d" % emb_w.shape[1]
        dims = dict(E=E, H=H, V=V)
        weights = dict(emb_w=emb_w, w_ih=ws[0], w_hh=ws[1], b_ih=ws[2], b_hh=ws[3], lin_w=ws[4], lin_b=ws[5])
        Desc, size_fn, run_fn, name = (_lib.BaseSampleDesc, "icd_baseline_sample_captions_ws_bytes",
                                       "icd_baseline_sample_captions", "icd_baseline_sample_captions")
    else:
        C = features.shape[-1]
        x = features.reshape(n_img, -1, C).contiguous().float()
        a = decoder.attention
        A, D, E, V = a.enc_att.weight.shape[0], decoder.decode_step.weight_hh.shape[1], \
            decoder.embedding.weight.shape[1], decoder.fc.weight.shape[0]
        emb_w = decoder.embedding.weight
        dims = dict(P=x.shape[1], C=C, A=A, D=D, E=E, V=V)
        weights = dict(enc_att_w=a.enc_att.weight, enc_att_b=a.enc_att.bias, dec_att_w=a.dec_att.weight,
                       dec_att_b=a.dec_att.bias, full_att_w=a.full_att.weight, full_att_b=a.full_att.bias,
                       w_ih=decoder.decode_step.weight_ih, w_hh=decoder.decode_step.weight_hh,
                       b_ih=decoder.decode_step.bias_ih, b_hh=decoder.decode_step.bias_hh,
                       h_lin_w=decoder.h_lin.weight, h_lin_b=decoder.h_lin.bias, c_lin_w=decoder.c_lin.weight,
                       c_lin_b=decoder.c_lin.bias, f_beta_w=decoder.f_beta.weight, f_beta_b=decoder.f_beta.bias,
                       fc_w=decoder.fc.weight, fc_b=decoder.fc.bias, emb_w=emb_w)
        Desc, size_fn, run_fn, name = _lib.SampleDesc, "icd_sample_captions_ws_bytes", "icd_sample_captions", \
            "icd_sample_captions"
    S1 = max_steps + 1
    groups = []
    ws_cache = None
    for j0 in range(0, n, 8):                             # samples in groups of at most 8, keyed by their global index
        m = min(8, n - j0)
        step_imgs = max(1, min(n_img, 65535 // m)) if chunk is None else int(chunk)
        g = dict(seq=torch.empty(n_img, m, S1 + 1, device=dev, dtype=torch.int32),
                 len=torch.empty(n_img, m, device=dev, dtype=torch.int32),
                 ended=torch.empty(n_img, m, device=dev, dtype=torch.uint8),
                 score=torch.empty(n_img, m, device=dev, dtype=torch.float32))
        if want_logp:
            g["logp"] = torch.empty(n_img, m, S1, device=dev, dtype=torch.float32)
        for i0 in range(0, n_img, step_imgs):
            ni = min(step_imgs, n_img - i0)
            d = Desc()
            fill(d, n_img=ni, m=m, max_steps=max_steps, precision=ops.precision_id(precision),
                 emb_is_f64=int(emb_w.dtype == torch.float64), start_id=start_id, end_id=end_id, top_k=int(top_k),
                 img_base=i0, sample_base=int(sample_base) + j0, temperature=float(temperature), seed=seed,
                 out_seq=g["seq"][i0:i0 + ni], out_len=g["len"][i0:i0 + ni], out_ended=g["ended"][i0:i0 + ni],
                 out_score=g["score"][i0:i0 + ni], out_logp=(g["logp"][i0:i0 + ni] if want_logp else None), **dims,
                 **weights)
            if base:
                fill(d, img_features=x[i0:i0 + ni])
            else:
                fill(d, enc=x[i0:i0 + ni])
            need = int(getattr(lib(), size_fn)(ctypes.byref(d)))
            if need < 0:
                check(-1, name)
            if ws_cache is None or ws_cache.numel() < need:
                ws_cache = torch.empty(need, device=dev, dtype=torch.uint8)
            d.ws = ws_cache.data_ptr()
            d.ws_bytes = need
            check(getattr(lib(), run_fn)(ctypes.byref(d), stream_ptr()), name)
        groups.append(g)
    out = {key: torch.cat([g[key] for g in groups], dim=1) for key in groups[0]}
    out["seed"] = seed
    return out


def beam_search_sharded(decoder, features_local, beam_size, start_id, end_id, max_steps=50, group=None, dst=0,
                        precision="fp32x3"):
    """BASELINE.json configs[4] / SURVEY.md 8e row 3: images are independent units, so every rank decodes its own shard
    with ``beam_search_batched`` (no collective during the decode) and ONE final gather brings caption lengths, token ids
    and scores to rank ``dst``.  All ranks must hold the same number of images.  Works unchanged in a single process.
    A ``BaselineDecoder`` takes (n, E) image features per rank and decodes with ``baseline_beam_search_batched``.
    -> on ``dst``: dict(len (world*n,), seq (world*n, max_steps+2), score (world*n,)) in rank order (CUDA tensors);
       elsewhere: None."""
    import torch.distributed as dist
    if isinstance(decoder, BaselineDecoder):
        res = baseline_beam_search_batched(decoder, features_local, beam_size, start_id, end_id, max_steps=max_steps,
                                           want_trace=False, precision=precision)
    else:
        res = beam_search_batched(decoder, features_local, beam_size, start_id, end_id, max_steps=max_steps,
                                  want_alphas=False, want_trace=False, precision=precision)
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        return {k: res[k] for k in ("len", "seq", "score")}
    world, rank = dist.get_world_size(group), dist.get_rank(group)
    n, S2 = res["seq"].shape
    # one packed int32 message per rank: [len | score bits | seq]
    packed = torch.cat([res["len"].view(n, 1), res["score"].view(torch.int32).view(n, 1), res["seq"]], dim=1).contiguous()
    parts = [torch.empty_like(packed) for _ in range(world)] if rank == dst else None
    dist.gather(packed, parts, dst=dst, group=group)
    if rank != dst:
        return None
    allp = torch.cat(parts, dim=0)
    return {"len": allp[:, 0].contiguous(), "score": allp[:, 1].contiguous().view(torch.float32), "seq": allp[:, 2:].contiguous()}


def attention_caption_image_beam_search(device, args, img, encoder, decoder, vocab):
    """Reads an image and captions it with beam search (gen_captions.py:16-131).

    Returns ``(seq, alphas, Caption_End)``: ``seq`` a python list of token ids including <start> and <end>,
    ``alphas`` a nested list (len(seq) x 14 x 14, first frame all ones), or ``([start, end], [], False)`` when no
    beam emitted <end> within the 51 steps the reference allows."""
    k = args.beam_size
    vocab_size = len(vocab)                                                         # :35
    encoder_out = encoder(img)                                                      # :37 (1, s, s, C)
    enc_image_size = encoder_out.size(1)
    start_id, end_id = vocab(START_TOKEN), vocab(END_TOKEN)
    with torch.no_grad():
        res = beam_search_batched(decoder, encoder_out, k, start_id, end_id, max_steps=50,
                                  want_alphas=True, want_trace=True)
    n = int(res["len"][0].item())
    trace = res["trace"][:, 0, :].tolist()
    for words in trace:                                                             # :91 per-step print
        live = [w for w in words if w >= 0]
        if not live:
            break
        print([vocab.i2w[w] for w in live])
    if n == 0:                                                                      # :123-125
        return [start_id, end_id], [], False
    seq = res["seq"][0, :n].tolist()
    alphas = res["alpha"][0, :n].view(n, enc_image_size, enc_image_size).tolist()
    assert vocab_size == decoder.fc.weight.shape[0]
    return seq, alphas, True


def baseline_caption_image_beam_search(device, args, img, encoder, decoder, vocab):
    """Captions an image with a ``BaselineDecoder`` — the counterpart of ``attention_caption_image_beam_search`` (same
    arguments, same per-step print of the candidate words) for the decoder the reference cannot generate with.

    ``encoder(img)`` returns the (1, E) image feature.  Returns ``(seq, Caption_End)``: ``seq`` a python list of token ids
    including <start> and <end>, or ``([start, end], False)`` when no beam emitted <end> within 51 steps.  Step 0 (the
    image feature) is not scored; position 0 is <start> (see the module docstring).  ``args.beam_size = 1`` is greedy."""
    k = args.beam_size
    features = encoder(img)
    start_id, end_id = vocab(START_TOKEN), vocab(END_TOKEN)
    with torch.no_grad():
        res = baseline_beam_search_batched(decoder, features.reshape(1, -1), k, start_id, end_id, max_steps=50,
                                           want_trace=True)
    n = int(res["len"][0].item())
    for words in res["trace"][:, 0, :].tolist():                                   # per-step print of the candidates
        live = [w for w in words if w >= 0]
        if not live:
            break
        print([vocab.i2w[w] for w in live])
    if n == 0:
        return [start_id, end_id], False
    assert len(vocab) == decoder.linear.weight.shape[0]
    return res["seq"][0, :n].tolist(), True
