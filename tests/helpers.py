"""Shared test helpers: seeded cases, digests, comparison utilities.

Every golden case is fully determined by a small dict of integers (dims + seeds): weights come from the module
constructors under ``torch.manual_seed`` (bit-identical between the reference and icd_b200 — asserted when the
goldens are generated and re-checked by checksum in the tests), inputs from ``icd_b200.synthetic``.
"""
import hashlib
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from icd_b200 import synthetic  # noqa: E402
from icd_b200.vocabulary import synthetic_vocab  # noqa: E402

GOLDEN_DIR = os.path.join(ROOT, "tests", "golden")

# name -> case description.  "full": whole tensors stored; "digest": norms + sampled entries stored.
ATT_CASES = {
    "att_small_ragged": dict(B=5, V=97, A=48, D=32, E=24, max_len=9, lengths=[9, 9, 7, 4, 2], wseed=0, iseed=11,
                             dropout=0.0, train=False, store="full", fine_tune_embedding=True),
    "att_small_unsorted": dict(B=4, V=97, A=48, D=32, E=24, max_len=8, lengths=[5, 8, 3, 8], wseed=1, iseed=12,
                               dropout=0.0, train=False, store="full", fine_tune_embedding=True, loss=False),
    "att_small_dropout": dict(B=4, V=97, A=48, D=32, E=24, max_len=7, lengths=[7, 7, 7, 7], wseed=2, iseed=13,
                              dropout=0.5, train=True, mask_seed=5, store="full", fine_tune_embedding=False),
    "att_cfg1": dict(B=4, V=9490, A=512, D=512, E=512, max_len=25, lengths=[25] * 4, wseed=0, iseed=1234,
                     dropout=0.0, train=False, store="digest", fine_tune_embedding=False),
    "att_glove": dict(B=3, V=211, A=64, D=64, E=300, max_len=10, lengths=[10, 8, 6], wseed=3, iseed=14,
                      dropout=0.0, train=False, store="digest", fine_tune_embedding=True, glove=True),
}
BASE_CASES = {
    "base_small": dict(B=6, V=97, E=32, H=32, L=9, wseed=0, iseed=21, store="full", lengths="ragged"),
    "base_cfg2": dict(B=128, V=9490, E=512, H=512, L=25, wseed=0, iseed=1234, store="digest", lengths=None),
}
BEAM_CASES = {
    # SURVEY.md 8c beam fixture recipe: embedding *= 30, fc.weight[END] *= gain, fc.bias[END] = bias
    "beam_cfg": dict(V=9490, A=512, D=512, E=512, k=5, wseed=0, iseed=77, n_img=6, emb_scale=30.0,
                     end_gain=30.0, end_bias=-4.0),
    "beam_small": dict(V=131, A=48, D=32, E=24, k=3, wseed=4, iseed=78, n_img=8, emb_scale=30.0,
                       end_gain=30.0, end_bias=-2.0),
}


def att_inputs(case):
    enc = synthetic.features(case["B"], seed=case["iseed"])
    caps, lens = synthetic.captions(case["B"], case["V"], max_len=case["max_len"], seed=case["iseed"],
                                    lengths=case["lengths"])
    return enc, caps, lens


def dropout_masks_like_reference(case, decode_lengths, D):
    """The keep-masks nn.Dropout draws inside the reference forward on CPU, in call order
    (one (batch_size_t, D) mask per step, models/attention.py:279), reproduced from the seed."""
    torch.manual_seed(case["mask_seed"])
    masks = []
    for t in range(max(decode_lengths)):
        bt = sum(l > t for l in decode_lengths)
        masks.append((torch.nn.functional.dropout(torch.ones(bt, D), case["dropout"], True) > 0).float())
    return masks


def stack_masks(masks, B, D):
    T = len(masks)
    out = torch.zeros(T, B, D, dtype=torch.uint8)
    for t, m in enumerate(masks):
        out[t, :m.shape[0]] = m.to(torch.uint8)
    return out


def build_attention_module(case, module_cls, params_cls, vocab, device="cpu"):
    p = params_cls()
    p.attention_dim, p.decoder_dim, p.embed_size = case["A"], case["D"], case["E"]
    p.dropout = case["dropout"]
    p.vocab = vocab
    torch.manual_seed(case["wseed"])
    dec = module_cls(torch.device(device), p)
    if case.get("glove"):
        dec.load_pretrained_embeddins(synthetic.glove_like_table(case["V"], case["E"]))
    dec.fine_tune_embeddings(case["fine_tune_embedding"])
    dec.train(case["train"])
    return dec


def build_baseline_module(case, module_cls, params_cls):
    p = params_cls()
    p.hidden_size, p.embed_size, p.vocab_size = case["H"], case["E"], case["V"]
    torch.manual_seed(case["wseed"])
    return module_cls(p)


def base_inputs(case):
    g = torch.Generator().manual_seed(case["iseed"])
    img = torch.randn(case["B"], case["E"], generator=g)
    caps, lens = synthetic.captions(case["B"], case["V"], max_len=case["L"], seed=case["iseed"],
                                    lengths=case["lengths"])
    return img, caps, lens


def apply_beam_recipe(dec, case):
    V = case["V"]
    with torch.no_grad():
        dec.embedding.weight *= case["emb_scale"]
        dec.fc.weight[V - 2] *= case["end_gain"]
        dec.fc.bias[V - 2] = case["end_bias"]


def beam_features(case):
    g = torch.Generator().manual_seed(case["iseed"])
    return torch.randn(case["n_img"], 14, 14, 2048, generator=g).abs()


# --------------------------------------------------------------------------------------------
def checksum(t):
    return hashlib.sha256(t.detach().cpu().contiguous().numpy().tobytes()).hexdigest()[:16]


def state_checksums(module):
    return {k: checksum(v) for k, v in module.state_dict().items()}


def sample_index(name, numel, n=48):
    seed = int(hashlib.sha256(name.encode()).hexdigest()[:8], 16)
    g = torch.Generator().manual_seed(seed)
    return torch.randint(0, numel, (min(n, numel),), generator=g)


def digest(name, t):
    t = t.detach().cpu().double().reshape(-1)
    idx = sample_index(name, t.numel())
    return dict(norm=float(t.norm()), sum=float(t.sum()), absmax=float(t.abs().max()),
                samples=t[idx].numpy().astype(np.float64))


def rel_err(a, b):
    a = a.detach().cpu().double()
    b = b.detach().cpu().double()
    den = float(b.norm())
    return float((a - b).norm()) / (den if den > 0 else 1.0)


def assert_close_norm(a, b, tol, what, atol=0.0):
    """Norm-wise relative comparison (SURVEY.md 8c caution (i)), with an absolute floor for tensors whose
    true value is ~0 (full_att.bias.grad)."""
    a = a.detach().cpu().double()
    b = b.detach().cpu().double()
    assert a.shape == b.shape, "%s: shape %s vs %s" % (what, tuple(a.shape), tuple(b.shape))
    err = float((a - b).norm())
    den = float(b.norm())
    assert err <= tol * den + atol, "%s: |a-b|=%.3e > %.1e*|b|(%.3e) + %.1e" % (what, err, tol, den, atol)


def assert_digest_close(name, t, dg, tol, atol=0.0):
    """Compare a tensor with a stored digest: norm, sum and the sampled entries."""
    t64 = t.detach().cpu().double().reshape(-1)
    idx = sample_index(name, t64.numel())
    norm = float(dg["norm"])
    assert abs(float(t64.norm()) - norm) <= tol * norm + atol, "%s: norm %.6e vs %.6e" % (name, float(t64.norm()), norm)
    s = torch.from_numpy(np.asarray(dg["samples"], dtype=np.float64))
    # sampled entries: error measured against the tensor's RMS scale, not the individual entry
    rms = norm / max(1.0, t64.numel() ** 0.5)
    err = float((t64[idx] - s).abs().max())
    assert err <= 20 * tol * rms + atol + tol * float(s.abs().max()), \
        "%s: sampled entries differ by %.3e (rms %.3e)" % (name, err, rms)


# --------------------------------------------------------------------------------------------
# fp64 oracle over a LARGE batch, evaluated in row chunks (rows are independent; only the parameters are shared), so
# the timed configuration (B = 512, V = 9490, full dimensions) can be checked tensor by tensor in about a minute.
# --------------------------------------------------------------------------------------------
def oracle_fp64_chunked(sd, enc, caps, lens, keep_mask=None, p=0.0, frozen=(), chunk=64, cuda_preds=None,
                        cuda_alphas=None, alpha_c=1.0, per_step=False, cuda_d_enc=None):
    """Full-batch loss and parameter gradients of the reference train step (models/attention.py:396-420) from the fp64
    oracle, accumulated over row chunks:  loss = sum_rows CE / n_packed + sum_{b,p} (alpha_c - sum_t alpha)^2 / (B*P).
    Lengths must be equal or sorted descending (then "first batch_size_t rows" == "rows with l > t" in every chunk).
    keep_mask: (T, B, D) uint8 dropout keep-mask (train mode) or None.
    cuda_preds / cuda_alphas: optional CPU fp32 copies of the CUDA outputs (or dicts name -> tensor for several candidates);
    their squared errors against the oracle are accumulated chunk by chunk.  -> dict(loss, grads{name: fp64}, err{predictions, alphas} norm-wise relative)
    Opt-in outputs (same candidate keying as ``err``):
      per_step=True -> step_sums{predictions, alphas}: (T, 2) fp64 [sum_b (got - ref)^2, sum_b ref^2] of every step t
        (all rows of the step; see step_rel_err);
      cuda_d_enc: candidate gradient(s) w.r.t. encoder_out, (B, ..., C) on any device (pulled to the host one row chunk at
        a time) -> row_sums: (B, 2) fp64 [|got_b - ref_b|^2, |ref_b|^2] per row (see row_rel_err).  The chunk's features
        are an fp64 leaf; the full fp64 reference gradient is never held."""
    from oracle import decoders as O
    import torch.nn.functional as F
    B = enc.shape[0]
    dl = [l - 1 for l in lens]
    assert all(dl[i] >= dl[i + 1] for i in range(B - 1)), "chunked oracle needs equal or descending lengths"
    T = max(dl)
    n_packed = sum(dl)
    C = enc.shape[-1]
    P = enc.reshape(B, -1, C).shape[1]
    w64 = {k: v.detach().cpu().double().clone().requires_grad_(k not in frozen) for k, v in sd.items()}
    loss_total = 0.0
    outputs = {}                      # candidate name -> (predictions, alphas) CPU tensors to be compared with the oracle
    if isinstance(cuda_preds, dict):
        outputs = {k: (cuda_preds[k], cuda_alphas[k]) for k in cuda_preds}
    elif cuda_preds is not None:
        outputs = {"": (cuda_preds, cuda_alphas)}
    denc = {}                         # candidate name -> gradient w.r.t. encoder_out
    if isinstance(cuda_d_enc, dict):
        denc = dict(cuda_d_enc)
    elif cuda_d_enc is not None:
        denc = {"": cuda_d_enc}
    acc = {k: {"predictions": [0.0, 0.0], "alphas": [0.0, 0.0]} for k in outputs}
    steps = {k: {"predictions": torch.zeros(T, 2, dtype=torch.float64), "alphas": torch.zeros(T, 2, dtype=torch.float64)}
             for k in outputs} if per_step else None
    rows = {k: torch.zeros(B, 2, dtype=torch.float64) for k in denc}
    margins, ids = [], []
    for r0 in range(0, B, chunk):
        r1 = min(B, r0 + chunk)
        if dl[r0] == 0:
            break
        ls = lens[r0:r1]
        masks = None
        if keep_mask is not None:
            masks = [keep_mask[t, r0:r0 + sum(1 for l in dl[r0:r1] if l > t)].double() for t in range(max(dl[r0:r1]))]
        e64 = enc[r0:r1].double().reshape(r1 - r0, P, C).requires_grad_(bool(denc))
        pr, _, dls, al = O.attention_decoder_forward(w64, e64, caps[r0:r1], ls, dropout_p=p,
                                                     dropout_masks=masks, hoist=True)
        Tc = max(dls)
        active = torch.tensor([[t < d for t in range(Tc)] for d in dls])
        tgt = caps[r0:r1, 1:Tc + 1]
        ce = F.cross_entropy(pr[active], tgt[active], reduction="sum") / n_packed
        reg = ((alpha_c - al.sum(dim=1)) ** 2).sum() / (B * P)
        (ce + reg).backward()
        loss_total += float(ce) + float(reg)
        with torch.no_grad():
            for cand, (c_pr, c_al) in outputs.items():
                for name, ref, got in (("predictions", pr, c_pr), ("alphas", al, c_al)):
                    gsl = got[r0:r1, :Tc].double()
                    acc[cand][name][0] += float(((gsl - ref) ** 2).sum())
                    acc[cand][name][1] += float((ref ** 2).sum())
                    if per_step:
                        steps[cand][name][:Tc, 0] += ((gsl - ref) ** 2).sum(dim=(0, 2))
                        steps[cand][name][:Tc, 1] += (ref ** 2).sum(dim=(0, 2))
            for cand, got in denc.items():
                g = got[r0:r1].detach().to("cpu", torch.float64).reshape(r1 - r0, P, C)
                rows[cand][r0:r1, 0] = ((g - e64.grad) ** 2).sum(dim=(1, 2))
                rows[cand][r0:r1, 1] = (e64.grad ** 2).sum(dim=(1, 2))
                del g
            e64 = None
            top2 = pr.detach().topk(2, dim=2)
            mg = torch.zeros(r1 - r0, T)
            ii = torch.zeros(r1 - r0, T, dtype=torch.int64)
            mg[:, :Tc] = (top2.values[..., 0] - top2.values[..., 1]).float()
            ii[:, :Tc] = top2.indices[..., 0]
            margins.append(mg)
            ids.append(ii)
    # rows of all-padding chunks contribute alpha_c^2 each to the regulariser (alphas stay 0)
    done_rows = min(B, ((max(i for i in range(B) if dl[i] > 0) // chunk) + 1) * chunk)
    loss_total += (B - done_rows) * P * alpha_c ** 2 / (B * P)
    # (their reference gradient w.r.t. the features is 0: the rows never attend and h0 / c0 are never used)
    for cand, got in denc.items():
        for r0 in range(done_rows, B, chunk):
            r1 = min(B, r0 + chunk)
            rows[cand][r0:r1, 0] = (got[r0:r1].detach().to("cpu", torch.float64).reshape(r1 - r0, -1) ** 2).sum(dim=1)
    err = {c: {k: ((v[0] ** 0.5) / (v[1] ** 0.5) if v[1] > 0 else None) for k, v in a.items()} for c, a in acc.items()}
    if list(err) == [""]:
        err = err[""]
    out = dict(loss=loss_total, grads={k: v.grad for k, v in w64.items() if v.grad is not None}, err=err,
               margin=torch.cat(margins, 0), ids=torch.cat(ids, 0), decode_lengths=dl)
    if per_step:
        out["step_sums"] = steps[""] if list(steps) == [""] else steps
    if denc:
        out["row_sums"] = rows[""] if list(rows) == [""] else rows
    return out


def step_rel_err(sums):
    """(T, 2) [squared error, squared reference] per step -> (T,) norm-wise relative error of each step (absolute where
    the reference is 0)."""
    return (sums[:, 0].sqrt() / torch.where(sums[:, 1] > 0, sums[:, 1], torch.ones_like(sums[:, 1])).sqrt())


row_rel_err = step_rel_err        # (B, 2) per-row sums -> (B,) relative error of each row


def aggregate_rel_err(sums):
    """Norm-wise relative error of the whole tensor from its per-step or per-row sums."""
    return float(sums[:, 0].sum().sqrt() / sums[:, 1].sum().sqrt())


def row_spread_failures(err_rows, bound, k):
    """Per-row criterion of the regime-B parity test: every row within ``bound`` and none more than ``k`` times the median
    row.  Rows are independent chains, so a row (or a group of rows) that some launch form computes wrongly stands out
    against the median even where the norm-wise error of the whole tensor hides it.  -> list of failure messages."""
    med = float(err_rows.median())
    bad = []
    worst = int(err_rows.argmax())
    if float(err_rows[worst]) > bound:
        over = (err_rows > bound).nonzero().flatten().tolist()
        bad.append("rows %s over the bound %.1e (worst row %d: %.2e)" % (over[:16], bound, worst, float(err_rows[worst])))
    if float(err_rows[worst]) > k * med:
        bad.append("row %d: %.2e > %g x the median row %.2e" % (worst, float(err_rows[worst]), k, med))
    return bad


def seeded_keep_mask(T, B, D, p, seed):
    g = torch.Generator().manual_seed(seed)
    return (torch.rand(T, B, D, generator=g) >= p).to(torch.uint8)
