"""Time of one self-critical sequence training (SCST) iteration per phase, both decoders, and of the weighted cross-entropy
gradient kernels against the unweighted ones on the same logits.

Iteration (the steps of ``scst.self_critical_loss``, written out so that CUDA events can sit between them): sample (m per
image, fp32x3, T = 1), greedy decode (the self-critical baseline), reward (word-fraction reward on the device; baseline and
advantage), pack and expand (``pack_samples``, ``features[img_idx]``), training forward (eval mode), loss (targets, weights,
``weighted_token_loss``), backward, optimiser (``DataParallelClipAdam``).  Cases:
  attention: 256 images x m = 5, 16-token cap (max_steps 15), V = 9490, A = D = E = 512, bf16 training tier with
             bf16_grad_only (as bench.py trains), fp32x3 sampling, greedy baseline;
  baseline : 1024 images x m = 5, same cap, E = H = 512, bf16 training tier.
Median over --reps iterations after --warmup, and the median of the whole ``self_critical_loss`` + backward + step timed the
same way, so that the written-out phases can be checked against the library call.

Kernels: the (R*T, 9490) logits of the attention case (R*T = 20 480 rows, 777 MB, more than the 126 MB L2), the unweighted and
weighted entry points alternated in one process, median of --kreps launches each: the streaming backward (fp32 + bf16
gradient) and the one-pass forward + bf16 gradient.  The card's name and power limit are read in the same run.  One JSON line
per case.

    python tools/scst_bench.py [--reps 10] [--warmup 3] [--kreps 30] [--out profiles/r06_scst_bench.jsonl]
"""
import argparse
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from baseline_beam_bench import gpu_info  # noqa: E402

PHASES = ["sample", "greedy", "reward", "pack_expand", "forward", "loss", "backward", "optimiser"]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--kreps", type=int, default=30)
    ap.add_argument("--max-steps", type=int, default=15)
    ap.add_argument("--m", type=int, default=5)
    ap.add_argument("--decoders", default="attention,baseline")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()

    import torch
    import __graft_entry__
    __graft_entry__.build()
    if not torch.cuda.is_available():
        raise SystemExit("scst_bench.py needs a CUDA device")
    import icd_b200.models.attention as my_att
    import icd_b200.models.baseline as my_base
    from icd_b200 import ops
    from icd_b200.gen_captions import sample_captions
    from icd_b200.losses import weighted_token_loss
    from icd_b200.parallel import DataParallelClipAdam
    from icd_b200.scst import baseline_rewards, pack_samples, scored_targets, self_critical_loss
    from icd_b200.vocabulary import synthetic_vocab

    V, E = 9490, 512
    dev = torch.device("cuda:0")
    start, end = V - 3, V - 2
    gen = torch.Generator().manual_seed(5)
    info = gpu_info()
    lines = []

    def reward(seq, ln):                       # fraction of a caption's words equal to token 7
        t = torch.arange(seq.shape[-1], device=seq.device)
        word = (t >= 1) & (t < ln[..., None]) & (seq != end)
        return (word & (seq == 7)).sum(-1).float() / word.sum(-1).clamp_min(1).float()

    def attention():
        p = my_att.AttentionDecoderParams()
        p.attention_dim, p.decoder_dim, p.embed_size = 512, 512, E
        p.vocab = synthetic_vocab(V)
        torch.manual_seed(0)
        dec = my_att.AttentionDecoder(dev, p)
        with torch.no_grad():
            dec.embedding.weight *= 30.0
            dec.fc.weight[V - 2] *= 30.0
            dec.fc.bias[V - 2] = -4.0
        feats = torch.randn(256, 196, 2048, generator=gen).abs().to(dev)
        return dec.to(dev), feats

    def baseline():
        p = my_base.BaselineDecoderParams()
        p.hidden_size, p.embed_size, p.vocab_size = 512, E, V
        torch.manual_seed(0)
        dec = my_base.BaselineDecoder(p)
        with torch.no_grad():
            dec.embedding.weight *= 30.0
            dec.linear.weight[V - 2] *= 15.0
            dec.linear.bias[V - 2] = -9.0
        feats = torch.randn(1024, E, generator=gen).to(dev)
        return dec.to(dev), feats

    m, S = a.m, a.max_steps
    saved_logits = {}
    for kind in a.decoders.split(","):
        dec, feats = attention() if kind == "attention" else baseline()
        base = kind == "baseline"
        dec.precision = "bf16"
        dec.train()
        grad_only = not base
        opt = DataParallelClipAdam(dec, lr=1e-6)
        n = feats.shape[0]

        def iteration(seed, ev):
            opt.zero_grad()
            ev[0].record()
            with torch.no_grad():
                s = sample_captions(dec, feats, m, start, end, seed=seed, max_steps=S, want_logp=True)
                ev[1].record()
                g = sample_captions(dec, feats, 1, start, end, temperature=0.0, seed=seed, max_steps=S)
                ev[2].record()
                r = reward(s["seq"], s["len"])
                adv = r - baseline_rewards(r, "greedy", reward(g["seq"], g["len"])[:, 0])
            ev[3].record()
            pk = pack_samples(s)
            x = feats[pk.img_idx]
            ev[4].record()
            was = dec.training
            dec.eval()
            logits = dec(x, pk.captions) if base else dec(x, pk.captions, pk.lengths)[0]
            dec.train(was)
            ev[5].record()
            tgt = scored_targets(pk.captions, pk.lengths, base, getattr(logits, "_icd_row_valid", None))
            w = pk.pack(adv)[:, None].expand(n * m, logits.shape[1]).contiguous()
            loss = weighted_token_loss(logits, tgt, w, sum(pk.lengths) - n * m, bf16_grad_only=grad_only)
            ev[6].record()
            loss.backward()
            ev[7].record()
            opt.step()
            ev[8].record()
            return pk, logits.shape

        def whole(seed, ev):
            opt.zero_grad()
            ev[0].record()
            loss, _ = self_critical_loss(dec, feats, reward, m, start, end, seed=seed, max_steps=S,
                                         bf16_grad_only=grad_only)
            loss.backward()
            opt.step()
            ev[1].record()

        per, tot, rows, steps = {p: [] for p in PHASES}, [], [], []
        for k in range(a.warmup + a.reps):
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(9)]
            pk, shape = iteration(100 + k, ev)
            torch.cuda.synchronize()
            if k >= a.warmup:
                for i, p in enumerate(PHASES):
                    per[p].append(ev[i].elapsed_time(ev[i + 1]))
                tot.append(ev[0].elapsed_time(ev[8]))
                rows.append(sum(pk.lengths) - len(pk.lengths))
                steps.append(shape[1])
        lib_ms = []
        for k in range(a.warmup + a.reps):
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
            whole(100 + k, ev)
            torch.cuda.synchronize()
            if k >= a.warmup:
                lib_ms.append(ev[0].elapsed_time(ev[1]))
        rec = dict(case="scst_iteration", decoder=kind, images=n, m=m, max_steps=S, V=V, training_tier="bf16",
                   bf16_grad_only=grad_only, sample_precision="fp32x3", baseline="greedy", reps=a.reps,
                   phase_ms_median={p: round(statistics.median(v), 3) for p, v in per.items()},
                   iteration_ms_median=round(statistics.median(tot), 3),
                   self_critical_loss_backward_step_ms_median=round(statistics.median(lib_ms), 3),
                   scored_tokens_median=int(statistics.median(rows)), train_steps_median=int(statistics.median(steps)),
                   gpu=info)
        print(json.dumps(rec), flush=True)
        lines.append(rec)
        del opt, dec, feats
        torch.cuda.empty_cache()

    # weighted vs unweighted kernels on the same logits (working set > L2)
    R = 256 * m * (S + 1)
    g = torch.Generator(device=dev).manual_seed(1)
    x = torch.randn(R, V, device=dev, generator=g) * 3.0
    t = torch.randint(0, V, (R,), device=dev, generator=g)
    t[::9] = -1
    w = torch.randn(R, device=dev, generator=g)
    up = torch.ones(1, device=dev)
    _, lse = ops.cross_entropy_fwd(x, t)
    calls = {
        "bwd_fp32_bf16": (lambda: ops.cross_entropy_bwd(x, t, lse, 1e-4, upstream=up, want_bf16=True),
                          lambda: ops.cross_entropy_bwd(x, t, lse, 1e-4, upstream=up, want_bf16=True, weights=w)),
        "fwd_grad16": (lambda: ops.cross_entropy_fwd_grad16(x, t, 1e-4),
                       lambda: ops.cross_entropy_fwd_grad16(x, t, 1e-4, weights=w)),
    }
    for name, (f0, f1) in calls.items():
        times = {0: [], 1: []}
        for k in range(3):
            f0(); f1()
        for k in range(a.kreps):
            for j, f in ((0, f0), (1, f1)) if k % 2 == 0 else ((1, f1), (0, f0)):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                f()
                e1.record()
                torch.cuda.synchronize()
                times[j].append(e0.elapsed_time(e1) * 1e3)
        u, wt = statistics.median(times[0]), statistics.median(times[1])
        rec = dict(case="ce_kernels", kernel=name, rows=R, V=V, logits_MB=round(R * V * 4 / 1e6, 1), launches_each=a.kreps,
                   unweighted_us_median=round(u, 1), weighted_us_median=round(wt, 1), weighted_over_unweighted=round(wt / u, 4),
                   gpu=info)
        print(json.dumps(rec), flush=True)
        lines.append(rec)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            for rec in lines:
                f.write(json.dumps(rec) + "\n")


if __name__ == "__main__":
    main()
