"""TEST INFRASTRUCTURE ONLY: self-critical sequence training (icd_b200.scst) restated on the CPU, in plain loops.

Inputs are the sampler's outputs for n images x m samples: ``seq`` (n, m, S) and ``len`` (n, m).
- ``pack``: R = n*m rows in a stable descending sort of the length (ties keep the flat index i*m + j); captions (R, Lmax) with
  0 beyond the length; lengths; the image and the flat index of each row.
- ``targets``: the scored positions of the training forward.  Attention decoder: t < len-1, target captions[r, t+1].
  Baseline decoder: 1 <= t <= len-1, target captions[r, t] (position 0 is the image step).  Either way these are the
  sampler's steps 1 .. len-1: attention position t is step t+1, baseline position t is step t.
- ``baseline_rewards``: "greedy" broadcasts the greedy caption's reward; "mean" is the leave-one-out mean (m >= 2).
- ``loss``: (1/N) sum over scored (r, t) of A_r * CE(logits[r, t], target), N the number of scored tokens.
"""
import torch
import torch.nn.functional as F


def pack(seq, ln):
    n, m = len(ln), len(ln[0])
    flat = [(i * m + j, int(ln[i][j])) for i in range(n) for j in range(m)]
    rows = sorted(flat, key=lambda x: -x[1])                       # Python's sort is stable
    perm = [k for k, _ in rows]
    lengths = [l for _, l in rows]
    Lmax = max(lengths)
    captions = torch.zeros(len(rows), Lmax, dtype=torch.int64)
    for r, (k, l) in enumerate(rows):
        for t in range(l):
            captions[r, t] = int(seq[k // m][k % m][t])
    return dict(captions=captions, lengths=lengths, img_idx=[k // m for k in perm], perm=perm)


def targets(captions, lengths, baseline_decoder):
    R, Lmax = captions.shape
    T = Lmax if baseline_decoder else Lmax - 1
    tgt = torch.full((R, T), -1, dtype=torch.int64)
    for r, l in enumerate(lengths):
        for t in range(T):
            if baseline_decoder and 1 <= t <= l - 1:
                tgt[r, t] = captions[r, t]
            elif not baseline_decoder and t < l - 1:
                tgt[r, t] = captions[r, t + 1]
    return tgt


def step_of(t, baseline_decoder):
    """The sampler step (1-based) that training position t scores."""
    return t if baseline_decoder else t + 1


def baseline_rewards(r, kind, greedy=None):
    n, m = r.shape
    b = torch.empty_like(r)
    for i in range(n):
        for j in range(m):
            if kind == "greedy":
                b[i, j] = greedy[i]
            else:
                b[i, j] = sum(float(r[i, k]) for k in range(m) if k != j) / (m - 1)
    return b


def loss(logits, tgt, adv_rows):
    """(R, T, V) logits, (R, T) targets, (R,) advantages in row order -> the SCST loss."""
    ce = F.cross_entropy(logits.reshape(-1, logits.shape[2]), tgt.reshape(-1).clamp_min(0), reduction="none").view(tgt.shape)
    scored = tgt >= 0
    return (adv_rows[:, None] * ce * scored).sum() / scored.sum()
