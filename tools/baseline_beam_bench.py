"""Time of the batched beam search over the BaselineDecoder (gen_captions.baseline_beam_search_batched ->
icd_baseline_beam_search): 1024 images x k = 5 at V = 9490, E = H = 512, fp32x3 — the workload bench.py's beam block runs
for the attention decoder, with the baseline's (n_img, E) image features instead of feature maps.

The decoder gets a beam fixture recipe (embedding x 30, linear.weight[<end>] x 15, linear.bias[<end>] = -9, cf. SURVEY.md 8c), so
captions end at realistic, varied lengths instead of running all 51 steps or ending at once; the length distribution is reported
with the time.  Median of --reps calls timed with CUDA events (after --warmup calls), captions/s,
and kernel launches per loop step (the library's launch counter: a call with max_steps = m minus one with m - 1).  One JSON line
per caption cap: max_steps 50 is the reference's cap (gen_captions.py:119), 24 the 25-token cap bench.py's attention beam
workload uses.

    python tools/baseline_beam_bench.py [--images 1024] [--k 5] [--reps 7] [--max-steps 50,24] [--out result.jsonl]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info():
    import torch
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=60)
        info["power_limit_and_max_sm_clock"] = q.stdout.strip()
    except (OSError, subprocess.SubprocessError):
        info["power_limit_and_max_sm_clock"] = "not read"
    return info


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--images", type=int, default=1024)
    ap.add_argument("--k", type=int, default=5)
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--precision", default="fp32x3")
    ap.add_argument("--max-steps", default="50,24")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()

    import torch
    import __graft_entry__
    __graft_entry__.build()
    if not torch.cuda.is_available():
        raise SystemExit("baseline_beam_bench.py needs a CUDA device")
    import icd_b200.models.baseline as my_base
    from icd_b200 import ops
    from icd_b200.gen_captions import baseline_beam_search_batched

    V, E, H = 9490, 512, 512
    dev = torch.device("cuda:0")
    p = my_base.BaselineDecoderParams()
    p.hidden_size, p.embed_size, p.vocab_size = H, E, V
    torch.manual_seed(0)
    dec = my_base.BaselineDecoder(p)
    with torch.no_grad():
        dec.embedding.weight *= 30.0
        dec.linear.weight[V - 2] *= 15.0
        dec.linear.bias[V - 2] = -9.0
    dec = dec.to(dev)
    feats = torch.randn(a.images, E, generator=torch.Generator().manual_seed(5)).to(dev)
    start, end = V - 3, V - 2

    def run(max_steps):
        with torch.no_grad():
            return baseline_beam_search_batched(dec, feats, a.k, start, end, max_steps=max_steps, precision=a.precision)

    gpu = gpu_info()
    lines = []
    for cap in [int(x) for x in a.max_steps.split(",")]:
        for _ in range(a.warmup):
            res = run(cap)
        torch.cuda.synchronize()
        times = []
        for _ in range(a.reps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            res = run(cap)
            e1.record()
            torch.cuda.synchronize()
            times.append(e0.elapsed_time(e1))
        n0 = ops.launch_count(); run(cap); torch.cuda.synchronize(); n_cap = ops.launch_count() - n0
        n0 = ops.launch_count(); run(cap - 1); torch.cuda.synchronize(); n_less = ops.launch_count() - n0
        lens = res["len"].cpu()
        done = lens[lens > 0].float()
        ms = statistics.median(times)
        lines.append(json.dumps({
            "workload": "baseline decoder beam search", "images": a.images, "k": a.k, "V": V, "E": E, "H": H,
            "precision": a.precision, "max_steps": cap, "max_caption_tokens": cap + 1,
            "median_ms": round(ms, 3), "min_ms": round(min(times), 3), "max_ms": round(max(times), 3), "reps": a.reps,
            "captions_per_s": round(a.images / (ms / 1e3), 1),
            "launches_per_call": n_cap, "launches_per_step": n_cap - n_less,
            "completed": int((lens > 0).sum()), "failed": int((lens == 0).sum()),
            "caption_len_mean": round(float(done.mean()), 2) if done.numel() else None,
            "caption_len_min_max": [int(done.min()), int(done.max())] if done.numel() else None,
            "gpu": gpu,
        }))
        print(lines[-1])
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
