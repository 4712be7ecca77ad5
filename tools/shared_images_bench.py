"""Captions that share images: the attention decoder's indexed training path (``forward(..., image_index=)``) against the
replicated one (``forward(features[img_idx], ...)``), alternated in one process.

Cases (one JSON line each, with the card's name and power limit read in the same run):
  scst       : the attention case of tools/scst_bench.py (256 images x m = 5, 16-token cap, V = 9490, A = D = E = 512, bf16
               training tier with bf16_grad_only, fp32x3 sampling, greedy baseline), median per phase over --reps iterations
               of each path; "pack" is pack_samples plus, on the replicated path, features[img_idx];
  teacher    : a teacher-forced bf16 train step (forward + loss + backward) on 100 images x 5 captions, lengths U{8..25};
  both cases : peak allocated memory of the training step (forward + loss + backward) of each path, and the attention-step
               forward / backward time from the library's icd_prof_* events (every 4th launch sampled; ms summed over the
               sampled launches of one step, the same launches on both paths).

    python tools/shared_images_bench.py [--reps 10] [--warmup 3] [--out profiles/r07_shared_images.jsonl]
"""
import argparse
import ctypes
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from baseline_beam_bench import gpu_info  # noqa: E402

PHASES = ["sample", "greedy", "reward", "pack", "forward", "loss", "backward", "optimiser"]
PATHS = ("indexed", "replicated")


def use(path):
    return path == "indexed"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--max-steps", type=int, default=15)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()

    import torch
    import __graft_entry__
    __graft_entry__.build()
    if not torch.cuda.is_available():
        raise SystemExit("shared_images_bench.py needs a CUDA device")
    import icd_b200.models.attention as my_att
    from icd_b200 import synthetic
    from icd_b200._lib import lib
    from icd_b200.gen_captions import sample_captions
    from icd_b200.losses import attention_caption_loss, weighted_token_loss
    from icd_b200.parallel import DataParallelClipAdam
    from icd_b200.scst import baseline_rewards, pack_samples, scored_targets
    from icd_b200.vocabulary import synthetic_vocab

    V, m, S = 9490, 5, a.max_steps
    dev = torch.device("cuda:0")
    start, end = V - 3, V - 2
    info = gpu_info()
    L = lib()
    lines = []

    def decoder():
        p = my_att.AttentionDecoderParams()
        p.attention_dim, p.decoder_dim, p.embed_size = 512, 512, 512
        p.vocab = synthetic_vocab(V)
        torch.manual_seed(0)
        dec = my_att.AttentionDecoder(dev, p)
        with torch.no_grad():
            dec.embedding.weight *= 30.0
            dec.fc.weight[V - 2] *= 30.0
            dec.fc.bias[V - 2] = -4.0
        dec = dec.to(dev)
        dec.precision = "bf16"
        return dec

    def prof(fn):
        """fn() once with every 4th attention-step launch timed -> (fwd_ms, bwd_ms) over the sampled launches."""
        fm, bm = ctypes.c_double(), ctypes.c_double()
        n = [ctypes.c_int64() for _ in range(4)]
        L.icd_prof_collect(ctypes.byref(fm), ctypes.byref(n[0]), ctypes.byref(n[1]), ctypes.byref(bm), ctypes.byref(n[2]),
                           ctypes.byref(n[3]))
        L.icd_prof_enable(4)
        fn()
        torch.cuda.synchronize()
        L.icd_prof_collect(ctypes.byref(fm), ctypes.byref(n[0]), ctypes.byref(n[1]), ctypes.byref(bm), ctypes.byref(n[2]),
                           ctypes.byref(n[3]))                  # (before switching off: that drops the recorded events)
        L.icd_prof_enable(0)
        return round(fm.value, 3), round(bm.value, 3)

    def peak(fn):
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats()
        base = torch.cuda.memory_allocated()
        fn()
        torch.cuda.synchronize()
        return round((torch.cuda.max_memory_allocated() - base) / 1e6, 1)

    # ---------------------------------------------------------------------------------------------------- SCST case
    dec = decoder()
    dec.train()
    opt = DataParallelClipAdam(dec, lr=1e-6)
    gen = torch.Generator().manual_seed(5)
    feats = torch.randn(256, 196, 2048, generator=gen).abs().to(dev)
    n = feats.shape[0]

    def reward(seq, ln):
        t = torch.arange(seq.shape[-1], device=seq.device)
        word = (t >= 1) & (t < ln[..., None]) & (seq != end)
        return (word & (seq == 7)).sum(-1).float() / word.sum(-1).clamp_min(1).float()

    def scst_train(pk, adv, indexed):
        dec.eval()
        if indexed:
            logits = dec(feats, pk.captions, pk.lengths, image_index=pk.img_idx_host)[0]
        else:
            logits = dec(feats[pk.img_idx], pk.captions, pk.lengths)[0]
        dec.train()
        tgt = scored_targets(pk.captions, pk.lengths, False, getattr(logits, "_icd_row_valid", None))
        w = pk.pack(adv)[:, None].expand(n * m, logits.shape[1]).contiguous()
        weighted_token_loss(logits, tgt, w, sum(pk.lengths) - n * m, bf16_grad_only=True).backward()

    def iteration(seed, ev, indexed):
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
        x = feats if indexed else feats[pk.img_idx]
        ev[4].record()
        dec.eval()
        logits = (dec(x, pk.captions, pk.lengths, image_index=pk.img_idx_host) if indexed else dec(x, pk.captions, pk.lengths))[0]
        dec.train()
        ev[5].record()
        tgt = scored_targets(pk.captions, pk.lengths, False, getattr(logits, "_icd_row_valid", None))
        w = pk.pack(adv)[:, None].expand(n * m, logits.shape[1]).contiguous()
        loss = weighted_token_loss(logits, tgt, w, sum(pk.lengths) - n * m, bf16_grad_only=True)
        ev[6].record()
        loss.backward()
        ev[7].record()
        opt.step()
        ev[8].record()
        return pk, adv

    per = {p: {ph: [] for ph in PHASES} for p in PATHS}
    tot = {p: [] for p in PATHS}
    for k in range(a.warmup + a.reps):
        for path in PATHS:                                   # the same seed (samples) on both paths, alternated
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(9)]
            pk, adv = iteration(100 + k, ev, use(path))
            torch.cuda.synchronize()
            if k >= a.warmup:
                for i, ph in enumerate(PHASES):
                    per[path][ph].append(ev[i].elapsed_time(ev[i + 1]))
                tot[path].append(ev[0].elapsed_time(ev[8]))
    pk, adv = iteration(999, [torch.cuda.Event() for _ in range(9)], True)
    mem = {p: peak(lambda: scst_train(pk, adv, use(p))) for p in PATHS}
    att = {p: prof(lambda: scst_train(pk, adv, use(p))) for p in PATHS}
    for path in PATHS:
        lines.append(dict(case="scst_iteration", path=path, images=n, m=m, max_steps=S, V=V, training_tier="bf16",
                          bf16_grad_only=True, sample_precision="fp32x3", baseline="greedy", reps=a.reps,
                          phase_ms_median={ph: round(statistics.median(v), 3) for ph, v in per[path].items()},
                          iteration_ms_median=round(statistics.median(tot[path]), 3),
                          train_step_peak_allocated_MB=mem[path],
                          att_step_ms_sampled_every_4th={"fwd": att[path][0], "bwd": att[path][1]}, gpu=info))
    del opt, dec, feats
    torch.cuda.empty_cache()

    # ------------------------------------------------------------------------------ teacher-forced, 100 images x 5 captions
    dec = decoder()
    dec.fine_tune_embeddings(False)
    dec.train()
    n_img, per_img = 100, 5
    B = n_img * per_img
    feats = synthetic.features(n_img, seed=3).to(dev)
    caps, lens = synthetic.captions(B, V, max_len=25, seed=4, lengths="ragged")
    caps = caps.to(dev)
    g = torch.Generator().manual_seed(6)
    idx = torch.randperm(B, generator=g) % n_img          # 5 captions per image, spread through the length-sorted batch
    idx_dev = idx.to(dev)

    def step(indexed):
        dec.zero_grad(set_to_none=True)
        if indexed:
            preds, _, dl, alphas = dec(feats, caps, lens, image_index=idx)
        else:
            preds, _, dl, alphas = dec(feats[idx_dev], caps, lens)
        attention_caption_loss(preds, caps, dl, alphas, bf16_grad_only=True).backward()

    times = {p: [] for p in PATHS}
    for k in range(a.warmup + a.reps):
        for path in PATHS:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.manual_seed(k)                          # the same dropout keep-mask on both paths
            e0.record()
            step(use(path))
            e1.record()
            torch.cuda.synchronize()
            if k >= a.warmup:
                times[path].append(e0.elapsed_time(e1))
    mem = {p: peak(lambda: step(use(p))) for p in PATHS}
    att = {p: prof(lambda: step(use(p))) for p in PATHS}
    for path in PATHS:
        lines.append(dict(case="teacher_forced_train_step", path=path, images=n_img, captions_per_image=per_img, rows=B,
                          lengths="U{8..25}", T=max(lens) - 1, V=V, training_tier="bf16", bf16_grad_only=True, reps=a.reps,
                          train_step_ms_median=round(statistics.median(times[path]), 3),
                          train_step_ms_min=round(min(times[path]), 3), train_step_peak_allocated_MB=mem[path],
                          att_step_ms_sampled_every_4th={"fwd": att[path][0], "bwd": att[path][1]}, gpu=info))
    out = open(a.out, "w") if a.out else None
    for ln in lines:
        s = json.dumps(ln)
        print(s)
        if out:
            out.write(s + "\n")
    if out:
        out.close()


if __name__ == "__main__":
    main()
