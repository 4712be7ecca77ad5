"""Time of seeded caption sampling (gen_captions.sample_captions -> icd_sample_captions / icd_baseline_sample_captions) next to
the beam search at k = m, both decoders: 1024 images x m = 5 samples at V = 9490, E = H = D = A = 512, fp32x3, temperature 1
with top_k in {0, 50}, caption caps of 25 and 51 tokens.

The decoders get the beam fixture recipe of tools/baseline_beam_bench.py (embedding x 30, the <end> row of the vocabulary layer
scaled, its bias lowered), so captions end at varied lengths.  Median of --reps calls timed with CUDA events (after --warmup
calls), samples/s, kernel launches per loop step (the library's launch counter: a call with max_steps = n minus one with n - 1),
the beam search at k = m timed the same way in the same process, and the card's name and power limit read in the same run.
One JSON line per (decoder, cap, top_k).  --profile F: instead, one sampler call and one beam call per decoder at the first cap
and top_k under torch.profiler (a run of its own), kernel time summed per kernel name, written to F as text.

    python tools/sample_bench.py [--images 1024] [--m 5] [--reps 7] [--max-steps 24,50] [--top-k 0,50] [--out result.jsonl]
    python tools/sample_bench.py --profile profile.txt
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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--images", type=int, default=1024)
    ap.add_argument("--m", type=int, default=5)
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--precision", default="fp32x3")
    ap.add_argument("--max-steps", default="24,50")
    ap.add_argument("--top-k", default="0,50")
    ap.add_argument("--decoders", default="baseline,attention")
    ap.add_argument("--out", default=None)
    ap.add_argument("--profile", default=None)
    a = ap.parse_args()

    import torch
    import __graft_entry__
    __graft_entry__.build()
    if not torch.cuda.is_available():
        raise SystemExit("sample_bench.py needs a CUDA device")
    import icd_b200.models.attention as my_att
    import icd_b200.models.baseline as my_base
    from icd_b200 import ops
    from icd_b200.gen_captions import baseline_beam_search_batched, beam_search_batched, sample_captions
    from icd_b200.vocabulary import synthetic_vocab

    V, E, H = 9490, 512, 512
    dev = torch.device("cuda:0")
    start, end = V - 3, V - 2
    gen = torch.Generator().manual_seed(5)

    def baseline():
        p = my_base.BaselineDecoderParams()
        p.hidden_size, p.embed_size, p.vocab_size = H, E, V
        torch.manual_seed(0)
        dec = my_base.BaselineDecoder(p)
        with torch.no_grad():
            dec.embedding.weight *= 30.0
            dec.linear.weight[V - 2] *= 15.0
            dec.linear.bias[V - 2] = -9.0
        feats = torch.randn(a.images, E, generator=gen).to(dev)
        return dec.to(dev), feats, baseline_beam_search_batched

    def attention():
        p = my_att.AttentionDecoderParams()
        p.attention_dim, p.decoder_dim, p.embed_size = 512, 512, E
        p.vocab = synthetic_vocab(V)
        torch.manual_seed(0)
        dec = my_att.AttentionDecoder(dev, p)
        dec.eval()
        with torch.no_grad():
            dec.embedding.weight *= 30.0
            dec.fc.weight[V - 2] *= 30.0
            dec.fc.bias[V - 2] = -4.0
        feats = torch.randn(a.images, 14, 14, 2048, generator=gen).abs().to(dev)
        beam = lambda *x, **kw: beam_search_batched(*x, want_alphas=False, **kw)          # noqa: E731
        return dec.to(dev), feats, beam

    def timed(fn):
        for _ in range(a.warmup):
            res = fn()
        torch.cuda.synchronize()
        times = []
        for _ in range(a.reps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            res = fn()
            e1.record()
            torch.cuda.synchronize()
            times.append(e0.elapsed_time(e1))
        return res, times

    def launches(fn, cap):
        n0 = ops.launch_count(); fn(cap); torch.cuda.synchronize(); n_cap = ops.launch_count() - n0
        n0 = ops.launch_count(); fn(cap - 1); torch.cuda.synchronize()
        return n_cap, n_cap - (ops.launch_count() - n0)

    gpu = gpu_info()
    if a.profile:
        from torch.profiler import ProfilerActivity, profile
        cap, top_k = int(a.max_steps.split(",")[0]), int(a.top_k.split(",")[0])
        report = ["GPU: %s" % json.dumps(gpu), "kernel time per call, %d images x m = k = %d, cap %d tokens, top_k %d, %s"
                  % (a.images, a.m, cap + 1, top_k, a.precision)]
        for name in a.decoders.split(","):
            dec, feats, beam = baseline() if name == "baseline" else attention()
            calls = (("sample", lambda: sample_captions(dec, feats, a.m, start, end, temperature=1.0, top_k=top_k, seed=1234,
                                                        max_steps=cap, precision=a.precision)),
                     ("beam", lambda: beam(dec, feats, a.m, start, end, max_steps=cap, precision=a.precision)))
            for what, fn in calls:
                with torch.no_grad():
                    fn(); fn(); torch.cuda.synchronize()
                    with profile(activities=[ProfilerActivity.CUDA]) as prof:
                        fn(); torch.cuda.synchronize()
                rows = sorted(((e.key, e.device_time_total / 1e3, e.count) for e in prof.key_averages() if e.device_time_total > 0),
                              key=lambda r: -r[1])
                total = sum(r[1] for r in rows)
                report.append("\n%s decoder, %s: %.3f ms kernel time" % (name, what, total))
                for k, ms, n in rows[:12]:
                    report.append("  %8.3f ms %5.1f %%  %5d x  %s" % (ms, 100 * ms / total, n, k[:110]))
            del dec, feats
            torch.cuda.empty_cache()
        os.makedirs(os.path.dirname(os.path.abspath(a.profile)), exist_ok=True)
        with open(a.profile, "w") as f:
            f.write("\n".join(report) + "\n")
        print("\n".join(report))
        return
    lines = []
    for name in a.decoders.split(","):
        dec, feats, beam = baseline() if name == "baseline" else attention()
        for cap in [int(x) for x in a.max_steps.split(",")]:
            with torch.no_grad():
                bres, btimes = timed(lambda: beam(dec, feats, a.m, start, end, max_steps=cap, precision=a.precision))
            for top_k in [int(x) for x in a.top_k.split(",")]:
                def samp(c, top_k=top_k):
                    with torch.no_grad():
                        return sample_captions(dec, feats, a.m, start, end, temperature=1.0, top_k=top_k, seed=1234,
                                               max_steps=c, precision=a.precision)
                res, times = timed(lambda: samp(cap))
                n_call, n_step = launches(samp, cap)
                lens = res["len"].float()
                ms, bms = statistics.median(times), statistics.median(btimes)
                lines.append(json.dumps({
                    "workload": "%s decoder caption sampling" % name, "images": a.images, "m": a.m, "V": V, "E": E, "H": H,
                    "precision": a.precision, "temperature": 1.0, "top_k": top_k, "max_steps": cap,
                    "max_caption_tokens": cap + 1,
                    "median_ms": round(ms, 3), "min_ms": round(min(times), 3), "max_ms": round(max(times), 3), "reps": a.reps,
                    "samples_per_s": round(a.images * a.m / (ms / 1e3), 1),
                    "launches_per_call": n_call, "launches_per_step": n_step,
                    "ended": int(res["ended"].sum()), "truncated": int((res["ended"] == 0).sum()),
                    "sample_len_mean": round(float(lens.mean()), 2),
                    "beam_k": a.m, "beam_median_ms": round(bms, 3), "beam_completed": int((bres["len"] > 0).sum()),
                    "gpu": gpu,
                }))
                print(lines[-1], flush=True)
        del dec, feats
        torch.cuda.empty_cache()
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
